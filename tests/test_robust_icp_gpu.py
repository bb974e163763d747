"""Row f11 (SURVEY.md §8f): Open3D's robust kernels for batched point-to-plane and generalized ICP on the GPU (csrc/icp.cu,
registration.icp / generalized_icp with kernel=...), against the numpy fp64 reference tests/robust_icp_oracle.py."""
import numpy as np
import pytest

import gicp_oracle as go
import robust_icp_oracle as ro
from test_gicp_gpu import _modelnet, _scan
from test_icp_gpu import _cuda, _pose_err
from test_robust_icp_oracle import (L2_MISS, OUTLIER_GICP_KERNEL, OUTLIER_PLANE_KERNEL, OUTLIER_R, OUTLIER_SEEDS,
                                    ROBUST_BOUND, moved_patch_scan)

pytestmark = pytest.mark.gpu

# k for point-to-plane in distance units; for generalized ICP in whitened units (distance / sqrt(2 eps) = 22 x distance along
# a shared normal at eps = 1e-3), gm in squared units of each
PLANE_KERNELS = ['l2', 'l1', ('huber', 0.01), ('cauchy', 0.01), ('gm', 1e-4), ('tukey', 0.05)]
GICP_KERNELS = ['l2', 'l1', ('huber', 0.2), ('cauchy', 0.2), ('gm', 0.04), ('tukey', 1.0)]
CASES = [(False, k) for k in PLANE_KERNELS] + [(True, k) for k in GICP_KERNELS]
_ID = lambda c: ('gicp-' if c[0] else 'plane-') + (c[1] if isinstance(c[1], str) else c[1][0])


def _loss(kernel):
    import ri_b200
    name, k = (kernel, 0.0) if isinstance(kernel, str) else kernel
    return ri_b200.ops.ROBUST_LOSSES.index(name), float(k)


def _robust(s, g, a, b, i0, r, gicp, kernel, eps=1e-3, max_iter=30, crit=1e-6, corr=True):
    """The robust op itself (also for 'l2', which registration routes to the plain estimators)."""
    import torch
    loss, k = _loss(kernel)
    T, fit, rmse, it, c = torch.ops.ri.robust_icp(s, g, a if gicp else None, b, i0, float(r), gicp, float(eps), loss, k,
                                                  max_iter, crit, crit, corr)
    return {'transformation': T, 'fitness': fit, 'inlier_rmse': rmse, 'iterations': it, 'correspondences': c}


def _tol(kernel, tol, gicp=False):
    """L1's w = 1/|r| amplifies the rounding differences between the kernel and the oracle on residuals near zero, so its
    poses are compared 10x looser.  Generalized ICP's L1 one step gets a further 10x: each correspondence has three
    world-axis rows of the whitened residual, some of them near zero, and there w reacts to W's closed form (from a = R n
    with the fp32 R, orthonormal to about 1e-7) differing from the oracle's eigh."""
    if kernel != 'l1':
        return tol
    return 100 * tol if gicp else 10 * tol


def _q32(src, T):
    """q = T s as the kernel computes it: fp32 fma chain from the fp32 T (fp32 products are exact in fp64)."""
    T = T.astype(np.float32).astype(np.float64)
    s = src.astype(np.float32).astype(np.float64)
    f = lambda x: x.astype(np.float32).astype(np.float64)
    return np.stack([f(f(T[k, 2] * s[:, 2] + f(T[k, 1] * s[:, 1] + f(T[k, 0] * s[:, 0]))) + T[k, 3]) for k in range(3)], 1)


def _one_step_oracle(src, tgt, ns, nt, r, gicp, kernel, init):
    """The oracle's one-step T.  For L1 it starts from the kernel's fp32 q (and the source normals rotated by init), so
    that 1/|r| sees the same residuals; otherwise from init in fp64."""
    if kernel != 'l1':
        return _oracle(src, tgt, ns, nt, r, gicp, kernel, init, 1, 0.0)[0]
    I = np.eye(4)
    U = _oracle(_q32(src, init), tgt, ns.astype(np.float64) @ init[:3, :3].T, nt, r, gicp, kernel, I, 1, 0.0)[0]
    return U @ init


def _oracle(src, tgt, ns, nt, r, gicp, kernel, init, max_iter, crit):
    if gicp:
        return ro.generalized_icp_normals(src, tgt, ns, nt, r, kernel, 1e-3, init, max_iter, crit, crit)
    return ro.icp_point_to_plane(src, tgt, nt, r, kernel, init, max_iter, crit, crit)


# ---------------------------------------------------------------------------------------------- 1. evaluation
@pytest.mark.parametrize("case", CASES, ids=_ID)
def test_result_is_evaluate_registration_of_returned_pose(case):
    import torch
    import ri_b200
    gicp, kernel = case
    src, tgt, ns, nt, G, init = _modelnet(3, seed=44)
    s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
    res = _robust(s, g, a, b, i0, 0.1, gicp, kernel)
    ev = ri_b200.registration.evaluate_registration(s, g, 0.1, res['transformation'])
    for key in ('correspondences', 'fitness', 'inlier_rmse'):
        assert torch.equal(res[key], ev[key]), key


# ---------------------------------------------------------------------------------------------- 2. identities
@pytest.mark.parametrize("fixture", ["modelnet", "scan"])
def test_l2_and_huge_huber_bit_identical_to_point_to_plane(fixture):
    import torch
    import ri_b200
    if fixture == "modelnet":
        src, tgt, ns, nt, G, init = _modelnet(4, seed=9, jitter=0.01)
    else:
        src, tgt, ns, nt, G, init = _scan(20000, seed=3, noise=0.005)
    s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
    want = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation='point_to_plane', tgt_normals=b,
                                    return_correspondences=True)
    l2 = _robust(s, g, a, b, i0, 0.1, False, 'l2')
    hub = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation='point_to_plane', tgt_normals=b,
                                   return_correspondences=True, kernel=('huber', 1e30))
    for got in (l2, hub):
        for key in want:
            assert torch.equal(got[key], want[key]), key


def test_gicp_l2_through_robust_op_matches_generalized_icp():
    import ri_b200
    src, tgt, ns, nt, G, init = _modelnet(3, seed=44)
    s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
    want = ri_b200.registration.generalized_icp(s, g, 0.1, init=i0, src_normals=a, tgt_normals=b)
    got = _robust(s, g, a, b, i0, 0.1, True, 'l2')
    compared = 0
    for p in range(3):
        if min(go.generalized_icp_normals(src[p], tgt[p], ns[p], nt[p], 0.1, 1e-3, init[p])[5]) < 1.0:
            continue
        compared += 1
        assert int(got['iterations'][p]) == int(want['iterations'][p])
        assert (got['transformation'][p] - want['transformation'][p]).abs().max().item() < 1e-5
    assert compared >= 2


# ---------------------------------------------------------------------------------------------- 3. against the oracle
def _fixtures():
    src, tgt, ns, nt, G, init = _modelnet(3, seed=44)
    yield "modelnet", src, tgt, ns, nt, init, 0.1
    src, tgt, ns, nt, G, init = _scan(20000, seed=4, noise=0.005)
    yield "scan", src, tgt, ns, nt, init, 0.1


@pytest.mark.parametrize("case", CASES, ids=_ID)
def test_one_step_matches_oracle(case):
    gicp, kernel = case
    for name, src, tgt, ns, nt, init, r in _fixtures():
        s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
        T = _robust(s, g, a, b, i0, r, gicp, kernel, max_iter=1, crit=0.0)['transformation'].cpu().numpy()
        for p in range(len(src)):
            want = _one_step_oracle(src[p], tgt[p], ns[p], nt[p], r, gicp, kernel, init[p].astype(np.float64))
            assert np.abs(T[p] - want).max() < _tol(kernel, 1e-6, gicp), (name, p, T[p], want)


@pytest.mark.parametrize("case", CASES, ids=_ID)
def test_full_run_matches_oracle(case):
    gicp, kernel = case
    src, tgt, ns, nt, G, init = _modelnet(3, seed=44)
    s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
    res = _robust(s, g, a, b, i0, 0.1, gicp, kernel, max_iter=30, crit=0.0)
    T = res['transformation'].cpu().numpy()
    compared = 0
    for p in range(3):
        want = _oracle(src[p], tgt[p], ns[p], nt[p], 0.1, gicp, kernel, init[p], 30, 0.0)
        if min(want[5]) < 1.0:
            continue
        compared += 1
        assert np.abs(T[p] - want[0]).max() < _tol(kernel, 1e-4), (p, T[p], want[0])
    assert compared >= 1


@pytest.mark.parametrize("seed", OUTLIER_SEEDS)
def test_outlier_fixture_meets_oracle_bounds(seed):
    import ri_b200
    src, tgt, ns, nt, G, init = moved_patch_scan(5000, seed)
    s, g, a, b, i0 = _cuda(*(x[None].astype(np.float32) for x in (src, tgt, ns, nt, init)))
    reg = ri_b200.registration
    for gicp in (False, True):
        if gicp:
            run = lambda k: reg.generalized_icp(s, g, OUTLIER_R, init=i0, src_normals=a, tgt_normals=b, kernel=k)
        else:
            run = lambda k: reg.icp(s, g, OUTLIER_R, init=i0, estimation='point_to_plane', tgt_normals=b, kernel=k)
        l2 = run(None)['transformation'][0].cpu().numpy()
        rob = run(OUTLIER_GICP_KERNEL if gicp else OUTLIER_PLANE_KERNEL)['transformation'][0].cpu().numpy()
        assert _pose_err(l2, G)[1] > L2_MISS
        rre, rte = _pose_err(rob, G)
        assert rre < ROBUST_BOUND[0] and rte < ROBUST_BOUND[1], (gicp, rre, rte)


# ---------------------------------------------------------------------------------------------- 4. edge cases
@pytest.mark.parametrize("gicp", [False, True])
def test_tukey_below_every_residual_keeps_init(gicp):
    import torch
    src, tgt, ns, nt, G, init = _modelnet(2, seed=3)
    s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
    res = _robust(s, g, a, b, i0, 0.1, gicp, ('tukey', 1e-30))
    assert torch.equal(res['transformation'], i0)
    assert (res['iterations'] == 1).all()


@pytest.mark.parametrize("gicp", [False, True])
def test_l1_on_identical_clouds_is_identity(gicp):
    import torch
    src, tgt, ns, nt, G, init = _modelnet(2, seed=5)
    eye = np.tile(np.eye(4, dtype=np.float32), (2, 1, 1))
    s, a, i0 = _cuda(src, ns, eye)
    res = _robust(s, s, a, a, i0, 0.1, gicp, 'l1')
    assert torch.equal(res['transformation'], i0)
    for key in ('fitness', 'inlier_rmse'):
        assert torch.isfinite(res[key]).all()
    assert (res['fitness'] == 1.0).all() and (res['inlier_rmse'] == 0.0).all()


def test_gicp_zero_and_non_finite_normals():
    src, tgt, ns, nt, G, init = _modelnet(2, seed=6)
    ns = ns.copy(); nt = nt.copy()
    ns[:, ::7] = 0.0; nt[:, ::5] = 0.0; ns[:, 3::11] = np.nan; nt[:, 2::13] = np.inf
    s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
    for kernel in (('cauchy', 0.2), ('tukey', 1.0)):
        T = _robust(s, g, a, b, i0, 0.1, True, kernel, max_iter=1, crit=0.0)['transformation'].cpu().numpy()
        assert np.isfinite(T).all()
        for p in range(2):
            want = ro.generalized_icp_normals(src[p], tgt[p], ns[p], nt[p], 0.1, kernel, 1e-3, init[p], 1, 0.0, 0.0)
            assert np.abs(T[p] - want[0]).max() < 1e-6, (p, kernel)


# ---------------------------------------------------------------------------------------------- 5. determinism, independence
@pytest.mark.parametrize("gicp", [False, True])
def test_deterministic_and_pairs_independent(gicp):
    import torch
    src, tgt, ns, nt, G, init = _modelnet(6, seed=21, jitter=0.01)
    s, g, a, b, i0 = _cuda(src, tgt, ns, nt, init)
    kernel = ('cauchy', 0.2) if gicp else ('cauchy', 0.01)
    x = _robust(s, g, a, b, i0, 0.1, gicp, kernel)
    y = _robust(s, g, a, b, i0, 0.1, gicp, kernel)
    for key in x:
        assert torch.equal(x[key], y[key]), key
    for p in range(6):
        sl = slice(p, p + 1)
        one = _robust(s[sl], g[sl], a[sl], b[sl], i0[sl], 0.1, gicp, kernel)
        for key in x:
            assert torch.equal(one[key][0], x[key][p]), (p, key)


# ---------------------------------------------------------------------------------------------- 6. wiring
def test_register_pairs_and_meter_take_the_kernel():
    import torch
    import ri_b200
    reg = ri_b200.registration
    src, tgt, ns, nt, G, init = _modelnet(4, seed=12, jitter=0.01)
    s, g, b = _cuda(src, tgt, nt)
    feat = torch.randn(4, 32, src.shape[1], device="cuda")
    icp_kw = {'max_correspondence_distance': 0.1, 'estimation': 'point_to_plane', 'tgt_normals': b,
              'kernel': ('tukey', 0.05)}
    T, inl, m = reg.register_pairs(feat, feat, s, g, func='kabsch', icp=icp_kw)
    T0, _, _ = reg.register_pairs(feat, feat, s, g, func='kabsch')
    want = reg.icp(s, g, init=T0, **icp_kw)['transformation']
    assert torch.equal(T, want)
    meter = reg.MeterModelNet40_registration('kabsch', icp=icp_kw)
    meter.update((feat, feat), (s, g, torch.from_numpy(G.astype(np.float32)).cuda()))
    assert set(meter.compute()) == {'succ', 'rre', 'rte', 'rmse', 'reg_time', 'rmse_succ'}


def test_errors():
    import torch
    import ri_b200
    reg = ri_b200.registration
    s = torch.rand(2, 64, 3, device="cuda"); n = torch.rand(2, 64, 3, device="cuda")
    eye = torch.eye(4, device="cuda")[None].repeat(2, 1, 1)
    plane = dict(estimation='point_to_plane', tgt_normals=n)
    for bad in ('huber', ('huber',), ('huber', 0.0), ('tukey', -1.0), ('cauchy', float('inf')), ('gm', float('nan')),
                ('l1', 1.0), ('welsch', 1.0), ('huber', 'x'), 3):
        with pytest.raises(ValueError):
            reg.icp(s, s, 0.1, kernel=bad, **plane)
        with pytest.raises(ValueError):
            reg.generalized_icp(s, s, 0.1, src_normals=n, tgt_normals=n, kernel=bad)
    for k in ('l2', 'l1', ('huber', 0.1)):
        with pytest.raises(ValueError):
            reg.icp(s, s, 0.1, kernel=k)                                  # point-to-point takes no kernel
    with pytest.raises(RuntimeError):
        reg.generalized_icp(s, s, 0.1, epsilon=0.0, src_normals=n, tgt_normals=n, kernel='l1')
    with pytest.raises(RuntimeError):
        reg.icp(s, s, 0.0, kernel='l1', **plane)
    op = torch.ops.ri.robust_icp
    with pytest.raises(RuntimeError):
        op(s, s, None, n, eye, 0.1, False, 1e-3, 6, 1.0, 30, 1e-6, 1e-6, False)           # unknown loss
    with pytest.raises(RuntimeError):
        op(s, s, None, n, eye, 0.1, False, 1e-3, 2, 0.0, 30, 1e-6, 1e-6, False)           # k <= 0
    with pytest.raises(RuntimeError):
        op(s, s, None, n, eye, 0.1, True, 1e-3, 1, 0.0, 30, 1e-6, 1e-6, False)            # no src_normals
    with pytest.raises(RuntimeError):
        op(s, s, n, n, eye, 0.1, True, float('nan'), 1, 0.0, 30, 1e-6, 1e-6, False)      # bad epsilon
    with pytest.raises(RuntimeError):
        op(s, s, None, n[:, :10], eye, 0.1, False, 1e-3, 1, 0.0, 30, 1e-6, 1e-6, False)   # normals shape
    with pytest.raises(RuntimeError):
        op(s, s, None, n, eye, 0.1, False, 1e-3, 1, 0.0, -1, 1e-6, 1e-6, False)           # max_iter
