"""CPU self-test of the ICP reference (tests/icp_oracle.py, row f5): it recovers a known pose, and its evaluation follows the
nearest-neighbour definition.  No GPU needed."""
import numpy as np
import pytest

import icp_oracle as ref


def _pose(rng, deg, trans):
    ax = rng.standard_normal(3); ax /= np.linalg.norm(ax)
    a = np.deg2rad(deg)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    T = np.eye(4); T[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    v = rng.standard_normal(3); T[:3, 3] = v / np.linalg.norm(v) * trans
    return T


def _planes(rng, n):
    """Three orthogonal patches (floor and two walls) with their normals: well-posed for both estimations."""
    k = n // 3
    p = rng.uniform(0, 1, (3 * k, 3)); nrm = np.zeros((3 * k, 3))
    for a in range(3):
        p[a * k:(a + 1) * k, a] = 0.0; nrm[a * k:(a + 1) * k, a] = 1.0
    return p, nrm


@pytest.mark.parametrize("estimation", ["point_to_point", "point_to_plane"])
def test_oracle_icp_recovers_known_pose(estimation):
    rng = np.random.default_rng(1)
    src, nrm = _planes(rng, 1500)
    G = _pose(rng, 20, 0.3)
    tgt = src @ G[:3, :3].T + G[:3, 3]
    tn = nrm @ G[:3, :3].T
    init = _pose(rng, 3, 0.03) @ G
    if estimation == "point_to_point":
        T, fit, rmse, it, corr = ref.icp_point_to_point(src, tgt, 0.1, init)
    else:
        T, fit, rmse, it, corr = ref.icp_point_to_plane(src, tgt, tn, 0.1, init)
    assert np.abs(T - G).max() < 1e-6
    assert fit == 1.0 and rmse < 1e-6 and 1 <= it < 30
    assert np.array_equal(corr, np.arange(len(src)))


def test_oracle_evaluate_matches_brute_force():
    rng = np.random.default_rng(2)
    src = rng.uniform(-1, 1, (300, 3)); tgt = rng.uniform(-1, 1, (500, 3))
    T = _pose(rng, 10, 0.1)
    r = 0.15
    fit, rmse, corr = ref.evaluate_registration(src, tgt, r, T)
    q = src @ T[:3, :3].T + T[:3, 3]
    d = np.linalg.norm(q[:, None] - tgt[None], axis=2)
    j = d.argmin(1); dm = d[np.arange(len(q)), j]
    want = np.where(dm < r, j, -1)
    assert np.array_equal(corr, want)
    assert fit == (dm < r).mean()
    assert abs(rmse - np.sqrt(np.mean(dm[dm < r] ** 2))) < 1e-12


def test_oracle_max_iter_zero_and_empty():
    rng = np.random.default_rng(3)
    src = rng.uniform(0, 1, (100, 3)); tgt = src + 10.0
    init = _pose(rng, 5, 0.05)
    T, fit, rmse, it, corr = ref.icp_point_to_point(src, tgt, 0.1, init, max_iter=0)
    assert np.array_equal(T, init) and it == 0 and fit == 0.0 and rmse == 0.0 and (corr == -1).all()
    T, fit, rmse, it, corr = ref.icp_point_to_plane(src, tgt, np.tile([0, 0, 1.0], (100, 1)), 0.1, init)
    assert np.array_equal(T, init) and it == 1 and fit == 0.0
