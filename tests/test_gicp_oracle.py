"""CPU self-test of tests/gicp_oracle.py, the fp64 reference that tests/test_gicp_gpu.py holds csrc/icp.cu's generalized
ICP (row f9) to: the covariance formula, the two forms of the update, the Jacobian, the eps = 1 limit, ground-truth
recovery and max_iter = 0."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import gicp_oracle as go
import icp_oracle


def _pose(rng, deg, trans):
    ax = rng.standard_normal(3); ax /= np.linalg.norm(ax)
    a = np.deg2rad(deg)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    T = np.eye(4); T[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    v = rng.standard_normal(3); T[:3, 3] = v / np.linalg.norm(v) * trans
    return T


def _pose_err(T, G):
    D = T[:3, :3] @ G[:3, :3].T
    s = min(1.0, np.linalg.norm(D - np.eye(3)) / (2 * np.sqrt(2)))
    return np.degrees(2 * np.arcsin(s)), np.linalg.norm(T[:3, 3] - G[:3, 3])


def _random_terms(rng, m, eps):
    q = rng.uniform(-1, 1, (m, 3)); t = q + rng.normal(0, 0.02, (m, 3))
    ns = rng.standard_normal((m, 3)); nt = rng.standard_normal((m, 3))
    R = _pose(rng, 20.0, 0.0)[:3, :3]
    Cs = go.covariances_from_normals(ns, eps)
    return q, t, R @ Cs @ R.T, go.covariances_from_normals(nt, eps)


def test_normals_covariance_equals_open3d_svd_path():
    """Open3D's no-normals path (20-NN covariance, SVD, singular values (1,1,eps)) builds I - (1-eps) n n^T from the
    smallest-eigenvalue direction, i.e. the normal estimate_normals(radius=inf, max_nn=20) returns.  Checked where that
    direction is well separated."""
    rng = np.random.default_rng(0)
    u, v = rng.uniform(-1, 1, (2, 3000))
    x = np.stack([u, v, 0.2 * np.sin(2 * u) * np.cos(3 * v)], 1) + rng.normal(0, 1e-3, (3000, 3))
    eps = 1e-3
    C = go.covariances_open3d_knn(x, eps)
    _, idx = cKDTree(x).query(x, k=20)
    nb = x[idx]; d = nb - nb.mean(1, keepdims=True)
    w, V = np.linalg.eigh(np.einsum('mki,mkj->mij', d, d) / 20)
    normals = V[:, :, 0]
    gap = (w[:, 1] - w[:, 0]) / w[:, 2]
    clear = gap > 0.05
    assert clear.mean() > 0.9
    N = go.covariances_from_normals(normals, eps)
    assert np.abs(C[clear] - N[clear]).max() < 1e-9
    # sign and length of the normal do not matter; zero and non-finite normals give the identity
    assert np.array_equal(go.covariances_from_normals(-normals, eps), N)
    assert np.abs(go.covariances_from_normals(3.5 * normals, eps) - N).max() < 1e-15
    bad = go.covariances_from_normals(np.array([[0.0, 0, 0], [np.nan, 0, 1], [np.inf, 0, 0]]), eps)
    assert np.array_equal(bad, np.broadcast_to(np.eye(3), (3, 3, 3)))


@pytest.mark.parametrize("eps", [1e-3, 0.1, 1.0])
def test_sqrt_form_equals_inverse_form(eps):
    rng = np.random.default_rng(1)
    q, t, Cs, Ct = _random_terms(rng, 500, eps)
    Hs, gs = go.moments(q, t, Cs, Ct, 'sqrt')
    Hi, gi = go.moments(q, t, Cs, Ct, 'inv')
    assert np.abs(Hs - Hi).max() <= 1e-12 * np.abs(Hi).max()
    assert np.abs(gs - gi).max() <= 1e-12 * np.abs(Hi).max()
    # M = 2I - (1-eps)(a a^T + b b^T): eigenvalues in [2 eps, 2]
    ev = np.linalg.eigvalsh(Ct + Cs)
    assert ev.min() >= 2 * eps * (1 - 1e-12) and ev.max() <= 2 * (1 + 1e-12)


def test_jacobian_matches_finite_differences():
    """With M held fixed, E(x) = sum (U(x) q - t)^T M^-1 (U(x) q - t) has gradient 2 g at x = 0."""
    rng = np.random.default_rng(2)
    q, t, Cs, Ct = _random_terms(rng, 200, 0.05)
    Minv = np.linalg.inv(Cs + Ct)
    _, g = go.moments(q, t, Cs, Ct, 'inv')

    def energy(x):
        ca, sa, cb, sb, cg, sg = np.cos(x[0]), np.sin(x[0]), np.cos(x[1]), np.sin(x[1]), np.cos(x[2]), np.sin(x[2])
        R = (np.array([[cg, -sg, 0], [sg, cg, 0], [0, 0, 1]]) @ np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
             @ np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]]))
        d = q @ R.T + x[3:] - t
        return np.einsum('mi,mij,mj->', d, Minv, d)

    h = 1e-6
    fd = np.array([(energy(h * e) - energy(-h * e)) / (2 * h) for e in np.eye(6)])
    assert np.abs(fd - 2 * g).max() <= 1e-6 * np.abs(g).max()


def test_eps_one_is_the_linearised_point_to_point_step():
    """eps = 1: C = I, M = 2I, and the step is the least-squares solution of J0 x = -d."""
    rng = np.random.default_rng(3)
    q, t, Cs, Ct = _random_terms(rng, 300, 1.0)
    assert np.abs(Cs + Ct - 2 * np.eye(3)).max() < 1e-15             # R I R^T: exact up to rounding
    H, g = go.moments(q, t, Cs, Ct, 'sqrt')
    J0 = go.jacobian0(q).reshape(-1, 6)
    x = np.linalg.lstsq(J0, -(q - t).reshape(-1), rcond=None)[0]
    assert np.abs(np.linalg.solve(H, -g) - x).max() < 1e-10


def _scan(n, seed):
    import ri_b200
    S = ri_b200.synth.make_scan(n, seed=seed)
    return S[:3].T.astype(np.float64), S[3:].T.astype(np.float64)


def _modelnet(seed):
    import ri_b200
    src, tgt, R, t = ri_b200.synth.make_pairs(1, 1024, seed=seed, jitter=0.0)
    return src[0, :3].T.astype(np.float64), src[0, 3:].T.astype(np.float64)


@pytest.mark.parametrize("cloud", ["scan", "modelnet"])
def test_noise_free_ground_truth_recovered(cloud):
    rng = np.random.default_rng(4)
    s, n = _scan(10000, 5) if cloud == "scan" else _modelnet(44)
    G = _pose(rng, 30.0, 0.5)
    t = s @ G[:3, :3].T + G[:3, 3]
    init = _pose(rng, 5.0, 0.05) @ G
    T, fit, rmse, iters, _, min_eig = go.generalized_icp_normals(s, t, n, n @ G[:3, :3].T, 0.1, 1e-3, init)
    rre, rte = _pose_err(T, G)
    assert rre < 1e-4 and rte < 1e-5, (rre, rte, iters)
    assert fit == 1.0 and rmse < 1e-5 and min(min_eig) > 1.0


def test_max_iter_zero_is_evaluate_registration():
    rng = np.random.default_rng(6)
    s, n = _modelnet(44)
    t = s + rng.normal(0, 0.02, s.shape)
    T0 = _pose(rng, 3.0, 0.03)
    T, fit, rmse, iters, corr, min_eig = go.generalized_icp_normals(s, t, n, n, 0.05, 1e-3, T0, max_iter=0)
    want = icp_oracle.evaluate_registration(s, t, 0.05, T0)
    assert np.array_equal(T, T0) and iters == 0 and min_eig == []
    assert fit == want[0] and rmse == want[1] and np.array_equal(corr, want[2])
