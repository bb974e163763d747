"""Row f5 (SURVEY.md §8f): batched ICP refinement and registration evaluation on the GPU (csrc/icp.cu), against the numpy /
scipy reference (tests/icp_oracle.py: Open3D's registration_icp / evaluate_registration restated in fp64)."""
import numpy as np
import pytest

import icp_oracle as ref

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- inputs
def _pose(rng, deg, trans):
    """A rigid motion of exactly `deg` degrees about a random axis and a translation of length `trans`."""
    ax = rng.standard_normal(3); ax /= np.linalg.norm(ax)
    a = np.deg2rad(deg)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    T = np.eye(4); T[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    v = rng.standard_normal(3); T[:3, 3] = v / np.linalg.norm(v) * trans
    return T


def _pose_err(T, G):
    """(rotation angle of T_R G_R^T in degrees, |t_T - t_G|); the chord form, which unlike acos of the trace does not
    amplify the rounding of an fp32 rotation."""
    D = np.asarray(T, np.float64)[:3, :3] @ np.asarray(G, np.float64)[:3, :3].T
    s = min(1.0, np.linalg.norm(D - np.eye(3)) / (2 * np.sqrt(2)))
    return np.degrees(2 * np.arcsin(s)), np.linalg.norm(np.asarray(T, np.float64)[:3, 3] - np.asarray(G, np.float64)[:3, 3])


def _modelnet_pairs(P, n, seed, jitter=0.001):
    """synth.make_pairs, point-major, with the GT pose perturbed by 5 degrees / 5 cm as the init."""
    import ri_b200
    src, tgt, R, t = ri_b200.synth.make_pairs(P, n, seed=seed, jitter=jitter)
    rng = np.random.default_rng(seed)
    G = np.tile(np.eye(4), (P, 1, 1)); G[:, :3, :3] = R; G[:, :3, 3] = t
    init = np.stack([_pose(rng, 5.0, 0.05) @ G[p] for p in range(P)])
    pm = lambda a: np.ascontiguousarray(a.transpose(0, 2, 1))
    return pm(src[:, :3]), pm(tgt[:, :3]), pm(tgt[:, 3:]), G, init.astype(np.float32)


def _scan_pair(n, seed, noise=0.0):
    """A planar indoor scan (synth.make_scan) and its copy under a known SE(3) (+ noise); init 3 degrees / 3 cm off."""
    import ri_b200
    rng = np.random.default_rng(seed)
    S = ri_b200.synth.make_scan(n, seed=seed)
    s = S[:3].T.astype(np.float64); nrm = S[3:].T.astype(np.float64)
    G = _pose(rng, 10.0, 0.2)
    t = s @ G[:3, :3].T + G[:3, 3] + rng.standard_normal(s.shape) * noise
    init = _pose(rng, 3.0, 0.03) @ G
    f = lambda a: np.ascontiguousarray(a[None], dtype=np.float32)
    return f(s), f(t), f(nrm @ G[:3, :3].T), G[None], f(init)


def _cuda(*arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


# ---------------------------------------------------------------------------------------------- 1. correspondences
def _check_evaluation(src, tgt, T, r):
    """GPU evaluate_registration against the oracle's on the source transformed by the fp32 rounding of T.  A differing
    correspondence must be a near-tie or lie at the threshold; fitness / rmse agree to within those."""
    import ri_b200
    s, g, Td = _cuda(src, tgt, T.astype(np.float32))
    res = ri_b200.registration.evaluate_registration(s, g, r, Td)
    corr = res['correspondences'].cpu().numpy(); fit = res['fitness'].cpu().numpy(); rmse = res['inlier_rmse'].cpu().numpy()
    for p in range(len(src)):
        Tp = T[p].astype(np.float32).astype(np.float64)
        ofit, ormse, ocorr = ref.evaluate_registration(src[p], tgt[p], r, Tp)
        q = src[p].astype(np.float64) @ Tp[:3, :3].T + Tp[:3, 3]
        bad = np.nonzero(corr[p] != ocorr)[0]
        for i in bad:
            a, b = corr[p, i], ocorr[i]
            if a >= 0 and b >= 0:
                da, db = np.linalg.norm(q[i] - tgt[p, a]), np.linalg.norm(q[i] - tgt[p, b])
                assert abs(da - db) < 1e-6, (p, i, a, b, da, db)
            else:
                d = np.linalg.norm(q[i] - tgt[p, max(a, b)])
                assert abs(d - r) < 1e-6, (p, i, a, b, d)
        n1 = src.shape[1]
        assert abs(fit[p] - ofit) <= len(bad) / n1 + 1e-12
        if len(bad) == 0:
            assert abs(rmse[p] - ormse) <= 1e-4 * max(ormse, 1e-3)
        else:
            assert abs(rmse[p] - ormse) <= 1e-3 * max(ormse, r)
    return corr, fit, rmse


@pytest.mark.parametrize("P,n1,n2", [(3, 1024, 1024), (2, 37, 5000), (1, 50000, 50000)])
def test_correspondences_match_oracle(P, n1, n2):
    import ri_b200
    rng = np.random.default_rng(n1 + n2)
    if n2 >= 5000:
        tgt = np.stack([ri_b200.synth.make_scan(n2, seed=10 + p)[:3].T for p in range(P)]).astype(np.float32)
        r = 0.1
    else:
        tgt = np.ascontiguousarray(ri_b200.synth.make_clouds(P, n2, seed=7)[:, :3].transpose(0, 2, 1))
        r = 0.05
    src = np.stack([tgt[p, rng.integers(0, n2, n1)] + rng.normal(0, r / 2, (n1, 3)) for p in range(P)]).astype(np.float32)
    T = np.stack([_pose(rng, 2.0, 0.02) for _ in range(P)])
    corr, fit, _ = _check_evaluation(src, tgt, T, r)
    assert 0.2 < fit.min() and fit.max() < 1.0                      # both found and unmatched points are exercised


def test_duplicated_and_coincident_targets():
    import ri_b200
    rng = np.random.default_rng(4)
    base = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
    tgt = np.concatenate([base, base])[None]                       # every target point twice: index i and i + 300
    src = (base + rng.normal(0, 0.01, base.shape)).astype(np.float32)[None]
    corr, fit, _ = _check_evaluation(src, tgt, np.eye(4)[None], 0.1)
    assert (corr[corr >= 0] < 300).all(), "equal distances must go to the lowest target index"
    assert fit[0] == 1.0
    same = np.full((1, 500, 3), 0.25, np.float32)                  # all target points coincident
    src = (0.25 + rng.uniform(-0.1, 0.1, (1, 200, 3))).astype(np.float32)
    s, g, I = _cuda(src, same, np.eye(4, dtype=np.float32)[None])
    res = ri_b200.registration.evaluate_registration(s, g, 0.1, I)
    within = np.linalg.norm(src[0].astype(np.float64) - 0.25, axis=1) < 0.1
    c = res['correspondences'].cpu().numpy()[0]
    assert (c[within] == 0).all() and (c[~within] == -1).all()
    assert abs(float(res['fitness'][0]) - within.mean()) <= 1.0 / 200


def test_sources_outside_target_box():
    import ri_b200
    rng = np.random.default_rng(5)
    tgt = rng.uniform(0, 1, (2, 400, 3)).astype(np.float32)
    src = (rng.uniform(0, 1, (2, 100, 3)) + np.array([3.0, -2.0, 0.5])).astype(np.float32)
    s, g, I = _cuda(src, tgt, np.tile(np.eye(4, dtype=np.float32), (2, 1, 1)))
    res = ri_b200.registration.evaluate_registration(s, g, 0.5, I)
    assert (res['fitness'].cpu().numpy() == 0).all() and (res['inlier_rmse'].cpu().numpy() == 0).all()
    assert (res['correspondences'].cpu().numpy() == -1).all()


# ---------------------------------------------------------------------------------------------- 2./3. ICP against the oracle and GT
# seed 44 draws shapes on which point-to-plane is well-posed (on a sphere it cannot fix a rotation about the centre)
@pytest.mark.parametrize("estimation", ["point_to_point", "point_to_plane"])
def test_icp_fixed_iterations_matches_oracle_and_gt(estimation):
    import ri_b200
    src, tgt, nrm, G, init = _modelnet_pairs(3, 1024, seed=44)
    r = 0.1
    s, g, n, i0 = _cuda(src, tgt, nrm, init)
    res = ri_b200.registration.icp(s, g, r, init=i0, estimation=estimation, tgt_normals=n, max_iter=30,
                                   relative_fitness=0.0, relative_rmse=0.0)
    T = res['transformation'].cpu().numpy()
    assert (res['iterations'].cpu().numpy() == 30).all()
    for p in range(3):
        if estimation == "point_to_point":
            want = ref.icp_point_to_point(src[p], tgt[p], r, init[p], 30, 0.0, 0.0)
        else:
            want = ref.icp_point_to_plane(src[p], tgt[p], nrm[p], r, init[p], 30, 0.0, 0.0)
        assert np.abs(T[p] - want[0]).max() < 1e-4, (p, T[p], want[0])
        assert abs(float(res['fitness'][p]) - want[1]) < 2e-3
        rre, rte = _pose_err(T[p], G[p])
        assert rre < 0.1 and rte < 1e-3, (p, rre, rte)


def test_point_to_plane_on_scans_converges_no_slower():
    import ri_b200
    src, tgt, nrm, G, init = _scan_pair(50000, seed=3)
    s, g, n, i0 = _cuda(src, tgt, nrm, init)
    out = {}
    for est in ("point_to_point", "point_to_plane"):
        res = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation=est, tgt_normals=n)
        T = res['transformation'].cpu().numpy()[0]
        rre, rte = _pose_err(T, G[0])
        assert rre < 0.1 and rte < 1e-3, (est, rre, rte)
        out[est] = int(res['iterations'][0])
    want = ref.icp_point_to_plane(src[0], tgt[0], nrm[0], 0.1, init[0])
    assert np.abs(T - want[0]).max() < 1e-4
    assert out["point_to_plane"] <= out["point_to_point"], out


# ---------------------------------------------------------------------------------------------- 4. convergence criteria
def test_identical_clouds_stay_put():
    import ri_b200
    c = ri_b200.synth.make_clouds(2, 1024, seed=9)
    s, n = _cuda(c[:, :3].transpose(0, 2, 1), c[:, 3:].transpose(0, 2, 1))
    I = _cuda(np.tile(np.eye(4, dtype=np.float32), (2, 1, 1)))[0]
    for est in ("point_to_point", "point_to_plane"):
        res = ri_b200.registration.icp(s, s, 0.05, init=I, estimation=est, tgt_normals=n)
        assert (res['transformation'] - I).abs().max().item() < 1e-6
        assert (res['fitness'].cpu().numpy() == 1.0).all()
        assert (res['iterations'].cpu().numpy() == 1).all()


def test_max_iter_zero_and_returned_correspondences():
    import torch
    import ri_b200
    src, tgt, nrm, G, init = _modelnet_pairs(3, 1024, seed=44)
    s, g, n, i0 = _cuda(src, tgt, nrm, init)
    ev = ri_b200.registration.evaluate_registration(s, g, 0.1, i0)
    r0 = ri_b200.registration.icp(s, g, 0.1, init=i0, max_iter=0, return_correspondences=True)
    assert torch.equal(r0['transformation'], i0) and (r0['iterations'] == 0).all()
    assert torch.equal(r0['fitness'], ev['fitness']) and torch.equal(r0['inlier_rmse'], ev['inlier_rmse'])
    assert torch.equal(r0['correspondences'], ev['correspondences'])
    for est in ("point_to_point", "point_to_plane"):
        res = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation=est, tgt_normals=n, return_correspondences=True)
        again = ri_b200.registration.evaluate_registration(s, g, 0.1, res['transformation'])
        assert torch.equal(res['correspondences'], again['correspondences'])
        assert torch.equal(res['fitness'], again['fitness']) and torch.equal(res['inlier_rmse'], again['inlier_rmse'])


# ---------------------------------------------------------------------------------------------- 5. degenerate inputs
def test_no_correspondences_keeps_init():
    import torch
    import ri_b200
    rng = np.random.default_rng(6)
    tgt = rng.uniform(0, 1, (2, 300, 3)).astype(np.float32)
    src = (tgt + 5.0).astype(np.float32)
    init = np.stack([_pose(rng, 4.0, 0.1) for _ in range(2)]).astype(np.float32)
    nrm = np.tile(np.array([0, 0, 1], np.float32), (2, 300, 1))
    s, g, n, i0 = _cuda(src, tgt, nrm, init)
    for est in ("point_to_point", "point_to_plane"):
        res = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation=est, tgt_normals=n)
        assert torch.equal(res['transformation'], i0)
        assert (res['fitness'].cpu().numpy() == 0).all() and (res['inlier_rmse'].cpu().numpy() == 0).all()


def test_point_to_plane_singular_system_is_identity_update():
    import torch
    import ri_b200
    rng = np.random.default_rng(7)
    # (a) five correspondences: J^T J has rank <= 5
    tgt = rng.uniform(0, 1, (1, 5, 3)).astype(np.float32)
    src = (tgt + 0.01).astype(np.float32)
    nrm = rng.standard_normal((1, 5, 3)); nrm /= np.linalg.norm(nrm, axis=2, keepdims=True)
    # (b) collinear points with one shared normal: rank 3
    line = np.linspace(0, 1, 50)[:, None] * np.array([1.0, 2.0, 0.5])
    tgt2 = line[None].astype(np.float32); src2 = (tgt2 + np.array([0, 0, 0.01])).astype(np.float32)
    nrm2 = np.tile(np.array([0, 0, 1.0]), (1, 50, 1))
    for a, b, c in ((src, tgt, nrm), (src2, tgt2, nrm2)):
        s, g, n = _cuda(a, b, c.astype(np.float32))
        I = torch.eye(4, device="cuda")[None]
        res = ri_b200.registration.icp(s, g, 0.2, init=I, estimation="point_to_plane", tgt_normals=n)
        assert torch.equal(res['transformation'], I)
        assert torch.isfinite(res['inlier_rmse']).all() and (res['fitness'].cpu().numpy() == 1).all()


def test_errors():
    import torch
    import ri_b200
    icp = ri_b200.registration.icp
    s = torch.rand(2, 64, 3, device="cuda"); n = torch.rand(2, 64, 3, device="cuda")
    with pytest.raises(RuntimeError):
        icp(s.cpu(), s.cpu(), 0.1)
    with pytest.raises(RuntimeError):
        icp(torch.rand(2, 64, 4, device="cuda"), s, 0.1)
    with pytest.raises(RuntimeError):
        icp(s, torch.rand(3, 64, 3, device="cuda"), 0.1)
    with pytest.raises(RuntimeError):
        icp(s, s, 0.1, init=torch.eye(3, device="cuda")[None].repeat(2, 1, 1))
    with pytest.raises(RuntimeError):
        icp(s, s, 0.1, estimation="point_to_plane", tgt_normals=n[:, :10])
    with pytest.raises(RuntimeError):
        icp(s, s, 0.0)
    with pytest.raises(RuntimeError):
        icp(s, s, 0.1, max_iter=-1)
    with pytest.raises(ValueError):
        icp(s, s, 0.1, estimation="generalized")
    with pytest.raises(ValueError):
        icp(s, s, 0.1, estimation="point_to_plane")
    with pytest.raises(RuntimeError):
        torch.ops.ri.icp(s, s, None, torch.eye(4, device="cuda")[None].repeat(2, 1, 1), 0.1, True, 30, 1e-6, 1e-6, False)


# ---------------------------------------------------------------------------------------------- 6./7. determinism, independence
@pytest.mark.parametrize("estimation", ["point_to_point", "point_to_plane"])
def test_deterministic_and_pairs_independent(estimation):
    import torch
    import ri_b200
    src, tgt, nrm, G, init = _modelnet_pairs(6, 1024, seed=21, jitter=0.01)
    s, g, n, i0 = _cuda(src, tgt, nrm, init)
    kw = dict(estimation=estimation, tgt_normals=n, return_correspondences=True)
    a = ri_b200.registration.icp(s, g, 0.1, init=i0, **kw)
    b = ri_b200.registration.icp(s, g, 0.1, init=i0, **kw)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    assert len(set(a['iterations'].tolist())) > 1, "pairs should converge at different iterations"
    for p in range(6):
        one = ri_b200.registration.icp(s[p:p + 1], g[p:p + 1], 0.1, init=i0[p:p + 1], estimation=estimation,
                                       tgt_normals=n[p:p + 1], return_correspondences=True)
        for k in a:
            assert torch.equal(one[k][0], a[k][p]), (p, k)


def test_scan_deterministic():
    import torch
    import ri_b200
    src, tgt, nrm, G, init = _scan_pair(50000, seed=8, noise=0.005)
    s, g, n, i0 = _cuda(src, tgt, nrm, init)
    a = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation="point_to_plane", tgt_normals=n, return_correspondences=True)
    b = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation="point_to_plane", tgt_normals=n, return_correspondences=True)
    for k in a:
        assert torch.equal(a[k], b[k]), k


# ---------------------------------------------------------------------------------------------- 8. meter
def test_meter_with_icp_refinement():
    import ri_b200
    rng = np.random.default_rng(12)
    P, n, C = 8, 1024, 64
    src, tgt, nrm, G, _ = _modelnet_pairs(P, n, seed=12, jitter=0.01)
    gt = G.astype(np.float32)
    # Weak descriptors, as a learned extractor gives them: a smooth function of the position in the source frame plus heavy
    # noise, so only ~100 mutual matches survive per pair and many of them pair a point with a spatial neighbour.  That
    # leaves RANSAC a coarse pose (a few tenths of a degree), which is what ICP on the full clouds refines.  With
    # near-exact descriptors the RANSAC refit over true partners is already optimal and ICP has nothing to add.
    W = 6.0 * rng.standard_normal((C, 3))
    back = np.einsum('pni,pij->pnj', tgt.astype(np.float64) - G[:, None, :3, 3], G[:, :3, :3])      # target in the source frame
    desc = np.sin(np.einsum('ci,pni->pcn', W, src)).astype(np.float32)
    desc2 = (np.sin(np.einsum('ci,pni->pcn', W, back)) + 1.0 * rng.standard_normal((P, C, n))).astype(np.float32)
    perm = np.stack([rng.permutation(n) for _ in range(P)])
    tgt_s = np.stack([tgt[p][perm[p]] for p in range(P)])
    desc2 = np.ascontiguousarray(np.stack([desc2[p][:, perm[p]] for p in range(P)]))
    base = ri_b200.registration.MeterModelNet40_registration('ransac')
    base.update((desc, desc2), (src, tgt_s, gt))
    ref = ri_b200.registration.MeterModelNet40_registration('ransac', icp={'max_correspondence_distance': 0.05})
    ref.update((desc, desc2), (src, tgt_s, gt))
    a, b = base.compute(), ref.compute()
    assert set(b) == set(a) == {'succ', 'rre', 'rte', 'rmse', 'reg_time', 'rmse_succ'}
    assert b['rre'] <= a['rre'] and b['rmse'] <= a['rmse'], (a, b)
