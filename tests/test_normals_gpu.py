"""Row f6 (SURVEY.md §8f): batched normal estimation on the GPU (csrc/normals.cu) against the k-NN it is defined by, the numpy /
scipy reference (tests/normals_oracle.py) and analytic normals."""
import numpy as np
import pytest

import normals_oracle as ref

pytestmark = pytest.mark.gpu

ROOM_CENTRE = np.array([2.0, 1.5, 1.25])


# ---------------------------------------------------------------------------------------------- inputs
def _modelnet(B, N, seed):
    """synth.make_clouds: xyz [B,3,N] f32 and the analytic normals [B,3,N]."""
    import ri_b200
    c = ri_b200.synth.make_clouds(B, N, seed=seed)
    return np.ascontiguousarray(c[:, :3]), np.ascontiguousarray(c[:, 3:])


def _scans(B, N, seed, noise=0.005):
    """synth.make_scan: xyz [B,3,N] f32 and the analytic normals (pointing into the room) [B,3,N]."""
    import ri_b200
    S = np.stack([ri_b200.synth.make_scan(N, seed=seed + b, noise=noise) for b in range(B)])
    return np.ascontiguousarray(S[:, :3]), np.ascontiguousarray(S[:, 3:])


def _cuda(*arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


def _lim(r):
    """The cut on the k-NN's squared distance: min(radius^2 in fp32, 10000)."""
    r = np.float32(r)
    return float(min(r * r, np.float32(10000.0)))


def _estimate(xyz, r, max_nn, camera=None, prior=None):
    import ri_b200
    return ri_b200.functional.estimate_normals(xyz, r, max_nn, camera=camera, prior=prior, return_counts=True)


def _pose(rng, deg, trans):
    """A rigid motion of exactly `deg` degrees about a random axis and a translation of length `trans`."""
    ax = rng.standard_normal(3); ax /= np.linalg.norm(ax)
    a = np.deg2rad(deg)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    T = np.eye(4); T[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    v = rng.standard_normal(3); T[:3, 3] = v / np.linalg.norm(v) * trans
    return T


def _pose_err(T, G):
    """(rotation angle of T_R G_R^T in degrees, |t_T - t_G|), chord form."""
    D = np.asarray(T, np.float64)[:3, :3] @ np.asarray(G, np.float64)[:3, :3].T
    s = min(1.0, np.linalg.norm(D - np.eye(3)) / (2 * np.sqrt(2)))
    return np.degrees(2 * np.arcsin(s)), np.linalg.norm(np.asarray(T, np.float64)[:3, 3] - np.asarray(G, np.float64)[:3, 3])


def _scan_pair(n, seed, noise):
    """A make_scan source [1,n,3], its copy under a known SE(3) plus noise, the analytic target normals, the pose and an init
    3 degrees / 3 cm off (point-major, as registration.icp takes them)."""
    import ri_b200
    rng = np.random.default_rng(seed)
    S = ri_b200.synth.make_scan(n, seed=seed)
    s = S[:3].T.astype(np.float64); nrm = S[3:].T.astype(np.float64)
    G = _pose(rng, 10.0, 0.2)
    t = s @ G[:3, :3].T + G[:3, 3] + rng.standard_normal(s.shape) * noise
    init = _pose(rng, 3.0, 0.03) @ G
    f = lambda a: np.ascontiguousarray(a[None], dtype=np.float32)
    return f(s), f(t), f(nrm @ G[:3, :3].T), G[None], f(init)


def _signed_angle(a, b):
    """Angle in radians between the rows of a and b, as atan2(|a x b|, a.b).  Unlike arccos of the dot product this neither
    needs unit rows nor amplifies their rounding: an fp32 normal is unit only to ~6e-8, which arccos near 1 would turn into
    an apparent angle of ~3e-4 rad."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.sum(a * b, 1))


def _angle(a, b):
    """Angle in radians between the rows of a and b, ignoring the sign."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.abs(np.sum(a * b, 1)))


# ---------------------------------------------------------------------------------------------- 1. neighbour selection
@pytest.mark.parametrize("workload", ["modelnet", "scan"])
def test_counts_equal_radius_cut_of_knn(workload):
    import ri_b200
    if workload == "modelnet":
        xyz, _ = _modelnet(32, 1024, seed=1)
        radii = (0.05, 0.2, float("inf"))
    else:
        xyz, _ = _scans(2, 50000, seed=2)
        radii = (0.05, 0.1, float("inf"))
    x, = _cuda(xyz)
    for max_nn in (1, 3, 8, 20, 30, 32):
        dist, _ = ri_b200.functional.knn_indices(x, max_nn)
        for r in radii:
            _, cnt = _estimate(x, r, max_nn)
            want = (dist < _lim(r)).sum(1).int()
            assert (cnt == want).all(), (workload, max_nn, r, int((cnt != want).sum()))
        assert int(cnt.min()) == max_nn                                 # radius = inf: plain k-NN


# ---------------------------------------------------------------------------------------------- 2. normals against the oracle
def _check_against_oracle(xyz, r, max_nn, camera=None, prior=None):
    """GPU normals vs the oracle on the k-NN's own neighbour lists, truncated by the radius."""
    import torch
    import ri_b200
    x, = _cuda(xyz)
    cam = None if camera is None else torch.from_numpy(np.asarray(camera, np.float32)).cuda()
    pri = None if prior is None else _cuda(prior)[0]
    nrm, cnt = _estimate(x, r, max_nn, camera=cam, prior=pri)
    dist, idx = ri_b200.functional.knn_indices(x, max_nn)
    want_cnt = (dist < _lim(r)).sum(1).int()
    assert torch.equal(cnt, want_cnt)
    nrm = nrm.cpu().numpy().astype(np.float64); cnt = cnt.cpu().numpy(); idx = idx.cpu().numpy()
    checked = 0
    for b in range(len(xyz)):
        p = xyz[b].T.astype(np.float64)
        cb = None if camera is None else np.asarray(camera, np.float32)[b].astype(np.float64)
        pb = None if prior is None else prior[b].T
        on, C, w = ref.normals_from_neighbours(p, idx[b].T, cnt[b], camera=cb, prior=pb)
        g = nrm[b].T
        assert np.abs(np.linalg.norm(g, axis=1) - 1).max() < 1e-6
        tr = np.trace(C, axis1=1, axis2=2)
        solved = (cnt[b] >= 3) & np.isfinite(tr) & (tr > 0)
        # degenerate neighbourhoods: the (0,0,1) default, oriented by the same rule
        assert np.array_equal(g[~solved], on[~solved]), b
        # everywhere: a near-minimal eigenvector
        q = np.einsum('ni,nij,nj->n', g, C, g)
        assert (q[solved] <= w[solved, 0] + 1e-6 * tr[solved]).all(), b
        # well-separated smallest eigenvalue: the same vector, and the same sign where the orientation test is decisive
        gap = solved & (w[:, 1] - w[:, 0] > 1e-3 * w[:, 2])
        ang = _angle(g[gap], on[gap])
        assert ang.max(initial=0.0) <= 1e-5, (b, ang.max())
        if camera is not None:
            dot = np.sum(on * (cb[None] - p), 1)
        elif prior is not None:
            dot = np.sum(on * pb, 1)
        else:
            dot = None
        if dot is not None:
            sure = gap & (np.abs(dot) > 1e-6)
            assert (np.sign(np.sum(g[sure] * on[sure], 1)) > 0).all(), b
        checked += int(gap.sum())
    return checked, cnt


@pytest.mark.parametrize("orient", ["camera", "prior", "none"])
def test_normals_match_oracle_modelnet(orient):
    xyz, truth = _modelnet(32, 1024, seed=3)
    kw = {"camera": np.tile([3.0, -2.0, 1.0], (32, 1))} if orient == "camera" else {"prior": truth} if orient == "prior" else {}
    # at radius 0.1 a 1024-point cloud of unit radius leaves many points with fewer than 3 neighbours (the default)
    for max_nn, r, share in ((30, 0.2, 0.7), (8, 0.1, 0.1), (32, float("inf"), 0.7)):
        checked, _ = _check_against_oracle(xyz, r, max_nn, **kw)
        assert checked > share * xyz.shape[0] * xyz.shape[2], (max_nn, r, checked)


@pytest.mark.parametrize("orient", ["camera", "prior"])
def test_normals_match_oracle_scans(orient):
    xyz, truth = _scans(2, 50000, seed=4)
    kw = {"camera": np.tile(ROOM_CENTRE, (2, 1))} if orient == "camera" else {"prior": truth}
    checked, _ = _check_against_oracle(xyz, 0.1, 30, **kw)
    assert checked > 0.9 * 2 * 50000, checked


# ---------------------------------------------------------------------------------------------- 3. independent search
def test_neighbour_sets_match_kdtree():
    """Against cKDTree in fp64: a set may differ only by a near-tie at the max_nn boundary or a point within 1e-6 of the
    radius (the GPU decides on fp32 squared distances)."""
    import ri_b200
    for xyz, r, max_nn in ((_modelnet(4, 1024, seed=5)[0], 0.05, 30), (_scans(1, 50000, seed=6)[0], 0.1, 30)):
        x, = _cuda(xyz)
        _, cnt = _estimate(x, r, max_nn)
        _, idx = ri_b200.functional.knn_indices(x, max_nn)
        cnt = cnt.cpu().numpy(); idx = idx.cpu().numpy()
        for b in range(len(xyz)):
            p = xyz[b].T.astype(np.float64)
            oidx, ocnt, _ = ref.hybrid_neighbours(p, r, max_nn)
            differ = 0
            for i in range(len(p)):
                mine, theirs = set(idx[b, :cnt[b, i], i].tolist()), set(oidx[i, :ocnt[i]].tolist())
                if mine == theirs:
                    continue
                differ += 1
                both = sorted(mine | theirs)
                edge = np.linalg.norm(p[both] - p[i], axis=1).max()          # the boundary of the fuller list
                full = max_nn in (len(mine), len(theirs))
                for j in mine ^ theirs:
                    d = np.linalg.norm(p[j] - p[i])
                    assert abs(d - r) < 1e-6 or (full and abs(d - edge) < 1e-6), (b, i, j, d, r, edge)
            assert differ <= 1e-3 * len(p), differ


# ---------------------------------------------------------------------------------------------- 4. ground truth
def test_noise_free_scan_planes_exact():
    import torch
    xyz, truth = _scans(1, 50000, seed=7, noise=0.0)
    x, = _cuda(xyz)
    cam = torch.tensor(ROOM_CENTRE, dtype=torch.float32, device="cuda")
    nrm, cnt = _estimate(x, 0.1, 30, camera=cam)
    import ri_b200
    _, idx = ri_b200.functional.knn_indices(x, 30)
    nrm = nrm.cpu().numpy()[0].T.astype(np.float64); cnt = cnt.cpu().numpy()[0]; idx = idx.cpu().numpy()[0]
    p = xyz[0].T; n = truth[0].T
    ax = np.abs(n).argmax(1)
    off = p[np.arange(len(p)), ax]
    # a neighbour is on the point's plane if it has the same analytic normal and the same (exact) offset along it
    same = np.ones(len(p), bool)
    for s in range(30):
        j = idx[s]
        use = s < cnt
        on = (np.abs(n[j] - n).sum(1) == 0) & (p[j, ax] == off)
        same &= ~use | on
    same &= cnt >= 3
    assert same.mean() > 0.7, same.mean()
    ang = _signed_angle(nrm[same], n[same])
    assert ang.max() <= 1e-5, ang.max()                     # signed: the camera sits inside the room


def test_noise_free_plane_and_sphere():
    import torch
    rng = np.random.default_rng(8)
    N, r = 4096, 0.15
    u = rng.standard_normal(3); u /= np.linalg.norm(u)
    e1 = np.cross(u, [0.0, 0.0, 1.0]); e1 /= np.linalg.norm(e1); e2 = np.cross(u, e1)
    uv = rng.uniform(-1, 1, (N, 2))
    plane = 0.2 * u + uv[:, :1] * e1 + uv[:, 1:] * e2
    s = rng.standard_normal((N, 3)); s /= np.linalg.norm(s, axis=1, keepdims=True)
    xyz = np.stack([plane.T, s.T]).astype(np.float32)
    cam = torch.tensor([[*(3.0 * u)], [0.0, 0.0, 0.0]], dtype=torch.float32, device="cuda")
    nrm, cnt = _estimate(_cuda(xyz)[0], r, 30, camera=cam)
    nrm = nrm.cpu().numpy().astype(np.float64)
    assert (cnt.cpu().numpy() >= 3).all()
    ang_plane = _signed_angle(nrm[0].T, np.tile(u, (N, 1)))     # signed: the camera is on the +u side
    assert ang_plane.max() <= 1e-5, ang_plane.max()
    pf = xyz[1].T.astype(np.float64); pf /= np.linalg.norm(pf, axis=1, keepdims=True)
    ang_sphere = _signed_angle(nrm[1].T, -pf)                   # camera at the centre: inward
    assert ang_sphere.max() <= np.arcsin(r) + 1e-5, ang_sphere.max()


# ---------------------------------------------------------------------------------------------- 5. degenerate inputs
def test_degenerate_inputs():
    import torch
    dev = "cuda"
    below = torch.tensor([0.0, 0.0, -10.0], device=dev)
    for N in (1, 2):
        x = torch.rand(3, 3, N, device=dev)
        nrm, cnt = _estimate(x, 10.0, 30, camera=below)
        assert (cnt == N).all() and (nrm == torch.tensor([0.0, 0.0, -1.0], device=dev)[None, :, None]).all()
    xyz, _ = _modelnet(3, 1024, seed=9)
    x, = _cuda(xyz)
    for max_nn in (1, 2):
        nrm, cnt = _estimate(x, 0.2, max_nn)
        assert (cnt <= max_nn).all() and (nrm == torch.tensor([0.0, 0.0, 1.0], device=dev)[None, :, None]).all()
    same = torch.full((2, 3, 500), 0.25, device=dev)
    nrm, cnt = _estimate(same, 0.1, 20)
    assert (cnt == 20).all() and (nrm == torch.tensor([0.0, 0.0, 1.0], device=dev)[None, :, None]).all()
    line_dir = np.array([1.0, 2.0, 0.5]); line_dir /= np.linalg.norm(line_dir)
    line = (np.sort(np.random.default_rng(10).uniform(0, 1, 300))[:, None] * line_dir).T[None].astype(np.float32)
    nrm, cnt = _estimate(_cuda(line)[0], 0.1, 20)
    g = nrm.cpu().numpy()[0].T.astype(np.float64)
    assert (cnt.cpu().numpy() >= 3).all()
    assert np.abs(np.linalg.norm(g, axis=1) - 1).max() < 1e-6 and np.abs(g @ line_dir).max() < 1e-5
    grid = np.stack(np.meshgrid(np.arange(10), np.arange(10), np.arange(10)), 0).reshape(1, 3, -1).astype(np.float32)
    nrm, cnt = _estimate(_cuda(grid)[0], 0.5, 30)                     # radius below the spacing: each point alone
    assert (cnt == 1).all() and (nrm == torch.tensor([0.0, 0.0, 1.0], device=dev)[None, :, None]).all()
    for shape in ((0, 3, 100), (4, 3, 0)):
        nrm, cnt = _estimate(torch.empty(shape, device=dev), 0.1, 30)
        assert tuple(nrm.shape) == shape and tuple(cnt.shape) == (shape[0], shape[2])


def test_errors():
    import torch
    import ri_b200
    en = ri_b200.functional.estimate_normals
    x = torch.rand(3, 3, 256, device="cuda")
    cam = torch.zeros(3, 3, device="cuda")
    for bad in (dict(max_nn=33), dict(max_nn=0), dict(radius=0.0), dict(radius=-1.0), dict(radius=float("nan")),
                dict(camera=cam, prior=x), dict(camera=torch.zeros(3, 2, device="cuda")),
                dict(camera=torch.zeros(4, 3, device="cuda")), dict(prior=x[:, :, :100].contiguous()),
                dict(prior=x[:2])):
        kw = dict(radius=0.1, max_nn=30); kw.update(bad)
        with pytest.raises(RuntimeError):
            en(x, kw.pop("radius"), **kw)
    with pytest.raises(RuntimeError):
        en(x.cpu(), 0.1)
    with pytest.raises(RuntimeError):
        en(x, 0.1, camera=cam.cpu())
    with pytest.raises(RuntimeError):
        en(torch.rand(3, 4, 256, device="cuda"), 0.1)


# ---------------------------------------------------------------------------------------------- 6. reproducibility
@pytest.mark.parametrize("B", [8, 5])
def test_deterministic_and_clouds_independent(B):
    import torch
    xyz, truth = _modelnet(B, 1024, seed=11)
    x, pr = _cuda(xyz, truth)
    for kw in (dict(), dict(prior=pr)):
        a = _estimate(x, 0.2, 30, **kw)
        b = _estimate(x, 0.2, 30, **kw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        for c in range(B):
            one = _estimate(x[c:c + 1], 0.2, 30, **{k: v[c:c + 1] for k, v in kw.items()})
            assert torch.equal(one[0][0], a[0][c]) and torch.equal(one[1][0], a[1][c]), c


def test_scans_deterministic():
    import torch
    xyz, _ = _scans(2, 50000, seed=12)
    x, = _cuda(xyz)
    cam = torch.tensor(ROOM_CENTRE, dtype=torch.float32, device="cuda")
    a = _estimate(x, 0.1, 30, camera=cam)
    b = _estimate(x, 0.1, 30, camera=cam)
    one = _estimate(x[1:], 0.1, 30, camera=cam)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(one[0][0], a[0][1]) and torch.equal(one[1][0], a[1][1])


# ---------------------------------------------------------------------------------------------- 7. integration with ICP
def test_point_to_plane_icp_with_estimated_normals():
    """An xyz-only scan pair: the target's normals estimated with the camera at the room centre drive point-to-plane ICP
    to ground truth, as the analytic normals do."""
    import torch
    import ri_b200
    src, tgt, nrm, G, init = _scan_pair(50000, seed=13, noise=0.005)
    s, g, n, i0 = _cuda(src, tgt, nrm, init)
    cam = torch.tensor(G[0, :3, :3] @ ROOM_CENTRE + G[0, :3, 3], dtype=torch.float32, device="cuda")
    est = ri_b200.functional.estimate_normals(g.transpose(1, 2).contiguous(), 0.1, 30, camera=cam)
    est = est.transpose(1, 2).contiguous()
    errs = {}
    for name, normals in (("estimated", est), ("analytic", n)):
        res = ri_b200.registration.icp(s, g, 0.1, init=i0, estimation="point_to_plane", tgt_normals=normals)
        errs[name] = _pose_err(res['transformation'].cpu().numpy()[0], G[0])
    rre, rte = errs["estimated"]
    assert rre < 0.05 and rte < 2e-3, errs
