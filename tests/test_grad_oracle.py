"""CPU checks of tests/grad_oracle.py, the fp64 restatements the GPU gradient tests compare against: each restated backward
against the C oracle's ri_oracle_*_grad (oracle/ri_oracle.c) and against the committed golden gradients (tests/golden/),
and each written-out backward against fp64 autograd of the restated forward.  Also the index range of the spherical grid
at r < 4, which is why the spherical devoxelizer refuses those resolutions."""
import ctypes

import numpy as np
import pytest
import torch

import grad_oracle as go
from _util import TOL, load_golden, rel_err, scaled_err


def D(a):
    return torch.from_numpy(np.ascontiguousarray(a)).double()


def I(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32))


def A(t):
    return t.detach().numpy()


def ball(rng, B, N):
    """Points in the unit ball, plus points the spherical grid leaves undefined: the origin, the south pole direction
    (beta = pi) and points at or beyond radius 1."""
    v = rng.standard_normal((B, 3, N))
    v *= rng.uniform(0.0, 1.0, (B, 1, N)) ** (1 / 3) / np.linalg.norm(v, axis=1, keepdims=True)
    v[:, :, 0] = 0.0
    v[:, :, 1] = (0.0, 0.0, -0.5)
    v[:, :, 2] = (1.0, 0.0, 0.0)
    v[:, :, 3] = (1.5, 0.0, 0.0)
    return v.astype(np.float32)


def autograd_vjp(fn, inputs, w):
    xs = [x.detach().double().requires_grad_(True) for x in inputs]
    return torch.autograd.grad(fn(*xs), xs, w)


# ====================================================================================================== k-NN
@pytest.mark.parametrize("c,n,m,k", [(3, 300, 200, 16), (5, 96, 64, 4), (1, 50, 40, 3), (3, 40, 5, 8)])
def test_knn_grad_matches_c_oracle(oracle, c, n, m, k):
    rng = np.random.default_rng(c * 1000 + n + k)
    x1 = rng.standard_normal((2, c, n)).astype(np.float32)
    x2 = rng.standard_normal((2, c, m)).astype(np.float32)
    x2[:, :, -2:] = x2[:, :, :2]                                          # duplicated references
    _, _, i1, i2 = oracle.knn(x1, x2, k)
    gd1 = rng.standard_normal((2, k, n)).astype(np.float32)
    gd2 = rng.standard_normal((2, k, m)).astype(np.float32)
    want = oracle.knn_grad(x1, x2, gd1, gd2, i1, i2)
    got = go.knn_grad(D(x1), D(x2), D(gd1), D(gd2), I(i1), I(i2))
    for g, w in zip(got, want):
        assert scaled_err(A(g), w) <= TOL


def test_knn_grad_golden(golden_dir):
    g = load_golden(golden_dir, "knn.npz")
    got = go.knn_grad(D(g["xyz1"]), D(g["xyz2"]), D(g["graddist1"]), D(g["graddist2"]), I(g["idx1"]), I(g["idx2"]))
    assert scaled_err(A(got[0]), g["gradxyz1"]) <= TOL and scaled_err(A(got[1]), g["gradxyz2"]) <= TOL


def test_knn_grad_sentinel_slots_and_skip_rule(oracle):
    """A query farther than 100 units from every reference has no neighbour under the forward's 10000 sentinel: all its slots
    hold (dist 10000, index 0).  The backward still differentiates those slots as distances to reference point 0, unless
    2 * graddist >= 20000 — the rule looks at the gradient, not the distance."""
    rng = np.random.default_rng(7)
    B, c, n, m, k = 1, 3, 6, 10, 4
    x1 = rng.standard_normal((B, c, n)).astype(np.float32)
    x1[0, :, 0] = (150.0, 0.0, 0.0)                                       # far query
    x2 = rng.standard_normal((B, c, m)).astype(np.float32)
    d1, d2, i1, i2 = oracle.knn(x1, x2, k)
    assert np.all(d1[0, :, 0] == 10000.0) and np.all(i1[0, :, 0] == 0)
    gd1 = np.ones((B, k, n), np.float32)
    gd1[0, :, 0] = (1.0, 9999.999, 10000.0, 25000.0)                      # the last two slots are skipped
    gd2 = np.zeros((B, k, m), np.float32)
    g1, g2 = go.knn_grad(D(x1), D(x2), D(gd1), D(gd2), I(i1), I(i2))
    w1, w2 = oracle.knn_grad(x1, x2, gd1, gd2, i1, i2)
    assert scaled_err(A(g1), w1) <= TOL and scaled_err(A(g2), w2) <= TOL
    diff = x1[0, :, 0].astype(np.float64) - x2[0, :, 0]
    assert np.allclose(A(g1)[0, :, 0], 2 * (1.0 + np.float64(np.float32(9999.999))) * diff, rtol=1e-12)
    only_far = go.knn_grad(D(x1[:, :, :1]), D(x2), D(gd1[:, :, :1]), D(gd2), I(i1[:, :, :1]), I(np.zeros_like(i2)))[1]
    assert np.allclose(A(only_far)[0, :, 0], -A(g1)[0, :, 0], rtol=1e-12)  # ... all of it lands on reference point 0
    assert not A(only_far)[0, :, 1:].any()


def test_knn_written_backward_equals_autograd_of_distances(oracle):
    rng = np.random.default_rng(3)
    x1 = rng.standard_normal((2, 5, 70)).astype(np.float32)
    x2 = rng.standard_normal((2, 5, 9)).astype(np.float32)
    _, _, i1, i2 = oracle.knn(x1, x2, 12)                                 # m < k: sentinel slots in dist1
    w1, w2 = D(rng.standard_normal((2, 12, 70))), D(rng.standard_normal((2, 12, 9)))
    want = autograd_vjp(lambda a, b: go.knn_dist(a, b, I(i1), I(i2)), (D(x1), D(x2)), (w1, w2))
    got = go.knn_grad(D(x1), D(x2), w1, w2, I(i1), I(i2))
    for g, w in zip(got, want):
        assert torch.allclose(g, w, rtol=1e-12, atol=1e-12)


# ================================================================================================== voxelize
@pytest.mark.parametrize("shape,r", [("spherical", 4), ("spherical", 8), ("spherical", 16), ("spherical", 32),
                                     ("cube", 4), ("cube", 8), ("cube", 16)])
def test_voxelize_grad_golden(golden_dir, shape, r):
    g = load_golden(golden_dir, "%s.npz" % shape)
    got = go.avg_voxelize_grad(D(g[f"r{r}_gy"]), I(g[f"r{r}_ind"]), I(g[f"r{r}_cnt"]))
    assert rel_err(A(got), g[f"r{r}_gx"]) <= TOL
    assert np.array_equal(A(got).astype(np.float32) == 0, g[f"r{r}_gx"] == 0)


@pytest.mark.parametrize("r", [2, 3, 5, 8])
def test_voxelize_grad_matches_c_oracle(oracle, r):
    rng = np.random.default_rng(r)
    B, C, N = 3, 7, 500
    pts = ball(rng, B, N)
    ind, cnt = oracle.sph_grid_stats(pts, r)
    assert (ind == -1).sum() >= 3 * B
    gy = rng.standard_normal((B, C, r ** 3)).astype(np.float32)
    want = oracle.avg_voxelize_grad(gy, ind, cnt)
    got = go.avg_voxelize_grad(D(gy), I(ind), I(cnt))
    assert rel_err(A(got), want) <= TOL
    # written-out backward == autograd of the restated means
    f = D(rng.standard_normal((B, C, N)))
    assert torch.equal(go.voxel_counts(I(ind), r ** 3), torch.from_numpy(cnt).long())
    (auto,) = autograd_vjp(lambda x: go.avg_voxelize(x, I(ind), r ** 3), (f,), D(gy))
    assert torch.allclose(got, auto, rtol=1e-14, atol=0)
    # ... and the restated means are the oracle's
    assert scaled_err(A(go.avg_voxelize(f, I(ind), r ** 3)), oracle.scatter_mean(A(f), ind, cnt, r)) <= TOL


# ================================================================================================ devoxelize
@pytest.mark.parametrize("shape,r", [("spherical", 4), ("spherical", 8), ("spherical", 16), ("spherical", 32),
                                     ("cube", 4), ("cube", 8), ("cube", 16)])
def test_devox_grad_golden(golden_dir, shape, r):
    g = load_golden(golden_dir, "%s.npz" % shape)
    got = go.devox_grad(D(g[f"r{r}_dgy"]), I(g[f"r{r}_dinds"]), D(g[f"r{r}_dwgts"]), r ** 3, shape == "spherical")
    assert scaled_err(A(got), g[f"r{r}_dgx"]) <= TOL
    # the forward through the same corners reproduces the golden devoxelized features
    grid = D(g[f"r{r}_grid"])
    assert scaled_err(A(go.devox(grid, I(g[f"r{r}_dinds"]), D(g[f"r{r}_dwgts"]))), g[f"r{r}_douts"]) <= TOL


@pytest.mark.parametrize("shape,r", [("spherical", 4), ("spherical", 7), ("cube", 2), ("cube", 9)])
def test_devox_grad_matches_c_oracle(oracle, shape, r):
    rng = np.random.default_rng(40 + r)
    B, C, N = 2, 9, 400
    grid = rng.standard_normal((B, C, r ** 3)).astype(np.float32)
    if shape == "spherical":
        pts = ball(rng, B, N)
        ind, _ = oracle.sph_grid_stats(pts, r)
        _, inds, wgts = oracle.spherical_trilinear_devoxelize(pts, grid, ind, r)
        assert (inds[:, 0] == -1).sum() >= B
    else:
        pts = (rng.uniform(0, r - 1, (B, 3, N))).astype(np.float32)
        pts[:, :, :40] = np.round(pts[:, :, :40])                          # on cell faces: zero high weights
        pts[:, 0, 40:60] = r - 1                                          # far face
        _, inds, wgts = oracle.trilinear_devoxelize(pts, grid, r)
    gy = rng.standard_normal((B, C, N)).astype(np.float32)
    want = oracle.devox_grad(gy, inds, wgts, r, shape == "spherical")
    got = go.devox_grad(D(gy), I(inds), D(wgts), r ** 3, shape == "spherical")
    assert scaled_err(A(got), want) <= TOL
    (auto,) = autograd_vjp(lambda x: go.devox(x, I(inds), D(wgts)), (D(grid),), D(gy))
    assert torch.allclose(got, auto, rtol=1e-12, atol=1e-12)


# ============================================================================================ edge / grouping
def test_edge_features_restatement(oracle):
    rng = np.random.default_rng(11)
    B, C, N, r = 2, 6, 300, 4
    pts = ball(rng, B, N)
    ind, cnt = oracle.sph_grid_stats(pts, r)
    f = rng.standard_normal((B, C, N)).astype(np.float32)
    avg = oracle.scatter_mean(f, ind, cnt, r)
    edge = go.voxel_edge_features(D(avg), D(f), I(ind))
    assert np.array_equal(A(edge).astype(np.float32), oracle.voxel_edge_gather(avg, f, ind))
    # its fp64 autograd: the relative half routes -g onto the point's cell and +g onto the point, neither for ind == -1
    w = D(rng.standard_normal((B, 2 * C, N)))
    g_avg, g_f = autograd_vjp(lambda a, x: go.voxel_edge_features(a, x, I(ind)), (D(avg), D(f)), w)
    keep = torch.from_numpy(ind != -1).unsqueeze(1).double()
    assert torch.equal(g_f, w[:, :C] * keep + w[:, C:])
    want_avg = torch.zeros(B, C, r ** 3, dtype=torch.float64)
    for b in range(B):
        for i in range(N):
            if ind[b, i] != -1:
                want_avg[b, :, ind[b, i]] -= w[b, :C, i]
    assert torch.allclose(g_avg, want_avg, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_grouping_grad_golden_and_oracle(golden_dir, oracle, case):
    g = load_golden(golden_dir, "ball_query.npz")
    idx = I(g[f"{case}_idx"])
    assert np.array_equal(A(go.grouping(D(g[f"{case}_feat"]), idx)).astype(np.float32), g[f"{case}_grp"])
    N = g[f"{case}_feat"].shape[2]
    got = go.grouping_grad(D(g[f"{case}_gy"]), idx, N)
    assert scaled_err(A(got), g[f"{case}_gx"]) <= TOL
    assert scaled_err(A(got), oracle.grouping_grad(g[f"{case}_gy"], g[f"{case}_idx"], N)) <= TOL
    (auto,) = autograd_vjp(lambda x: go.grouping(x, idx), (D(g[f"{case}_feat"]),), D(g[f"{case}_gy"]))
    assert torch.allclose(got, auto, rtol=1e-12, atol=1e-12)


# ===================================================================================== spherical grid at r < 4
@pytest.mark.parametrize("r", [2, 3, 4, 5])
def test_spherical_cells_stay_in_grid_but_devox_corners_do_not_below_r4(oracle, r):
    """The spherical voxelizer's cells stay inside the r^3 grid at every r, so it needs no guard.  The devoxelizer's corner
    rows are radians truncated to ints (the reference's quirk): its highest corner index is r^2 + 7r + 4, past r^3 for
    r = 2 and 3 — which is why ri_sph_trilinear_devox_f32 refuses r < 4."""
    rng = np.random.default_rng(100 + r)
    B, N = 2, 4000
    pts = ball(rng, B, N)
    ind, cnt = oracle.sph_grid_stats(pts, r)
    assert ind.min() == -1 and ind.max() < r ** 3 and int(cnt.sum()) == int((ind >= 0).sum())
    # corner indices straight from the C oracle, with a feature buffer long enough for any of them
    feat = np.zeros((r * r + 7 * r + 5,), np.float32)
    outs = np.empty((B, 1, N), np.float32)
    inds = np.empty((B, 8, N), np.int32)
    wgts = np.empty((B, 8, N), np.float32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    oracle.lib().ri_oracle_sph_trilinear_devox(P(pts), P(feat), P(ind), 1, 1, N, r, P(outs), P(inds), P(wgts))
    oracle.lib().ri_oracle_sph_trilinear_devox(P(pts[1:]), P(feat), P(ind[1:]), 1, 1, N, r, P(outs[1:]), P(inds[1:]),
                                               P(wgts[1:]))
    assert inds.max() <= r * r + 7 * r + 4
    beyond = int(((inds >= r ** 3) & (wgts != 0)).sum())
    assert (beyond > 0) == (r < 4), beyond
