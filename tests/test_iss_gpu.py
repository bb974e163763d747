"""Row f13 (SURVEY.md §8f): batched ISS keypoints on the GPU (csrc/iss.cu) against the numpy replay of the contract
(tests/iss_oracle.py), rigid-motion invariance, reproducibility, degenerate inputs, argument errors, the padding of
keypoint_batch, and the chain normals -> FPFH -> ISS -> keypoint_batch -> mutual_nn -> pose -> ICP."""
import ctypes
import math

import numpy as np
import pytest

import iss_oracle as O

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- helpers
def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _iss(xyz_cm, rs=0.0, rnm=0.0, **kw):
    """GPU ISS of a [B,3,N] batch -> (list of keypoint arrays, idx, count, saliency, radii) as numpy."""
    import ri_b200
    idx, cnt, sal, rad = ri_b200.functional.compute_iss_keypoints(xyz_cm, rs, rnm, return_saliency=True,
                                                                  return_radii=True, **kw)
    idx, cnt, sal, rad = idx.cpu().numpy(), cnt.cpu().numpy(), sal.cpu().numpy(), rad.cpu().numpy()
    return [idx[b, :cnt[b]] for b in range(len(cnt))], idx, cnt, sal, rad


def _compare(X, got_kp, got_sal, got_rad, rs=0.0, rnm=0.0, **kw):
    """One cloud X [N,3] against the oracle; -> (points compared, ambiguous points)."""
    o = O.iss(X, rs, rnm, **kw)
    amb = o['amb']
    if rs == 0.0 or rnm == 0.0:
        for g, w in zip(got_rad, o['radii']):
            assert abs(float(g) - float(w)) <= float(np.spacing(np.float32(w))), (got_rad, o['radii'])
    else:
        assert np.array_equal(got_rad, np.float32([rs, rnm]))
    assert np.all(np.diff(got_kp) > 0)
    mine = np.zeros(len(X), bool); mine[got_kp] = True
    want = np.zeros(len(X), bool); want[o['idx']] = True
    assert np.array_equal(mine[~amb], want[~amb]), (int((mine != want)[~amb].sum()), np.flatnonzero((mine != want) & ~amb)[:8])
    scale = np.abs(o['e1'])
    clear = ~amb
    err = np.abs(got_sal - o['saliency'])[clear]
    assert np.all(err <= 1e-9 * np.maximum(scale[clear], 1e-300) + 1e-300), err.max()
    return int(clear.sum()), int(amb.sum())


def _modelnet(B, N, seed):
    import ri_b200
    return np.ascontiguousarray(ri_b200.synth.make_clouds(B, N, seed=seed)[:, :3])


def _scans(S, N, seed):
    import ri_b200
    return np.stack([ri_b200.synth.make_scan(N, seed=seed + s)[:3] for s in range(S)])


# ---------------------------------------------------------------------------------------------- 1. the oracle
@pytest.mark.parametrize("case", ["modelnet_auto", "modelnet_explicit", "scan_auto", "scan_explicit", "fps_scan_auto"])
def test_keypoints_equal_oracle(case):
    import torch
    import ri_b200
    kw = {}
    rs = rnm = 0.0
    if case.startswith("modelnet"):
        xyz = _modelnet(16, 1024, seed=11)
        if case.endswith("explicit"):
            rs, rnm, kw = 0.15, 0.1, dict(min_neighbors=8, gamma_21=0.9, gamma_32=0.8)
    elif case.startswith("scan"):
        xyz = _scans(2, 50000, seed=3)
        if case.endswith("explicit"):
            rs, rnm = 0.1, 0.07
    else:
        scans = [torch.from_numpy(ri_b200.synth.make_scan(50000, seed=20 + s)[:3].T.copy()).cuda() for s in range(3)]
        subs = ri_b200.grid_sub_sampling_many(scans, grid_size=0.05)
        pts, _, _ = ri_b200.farthest_point_batch(subs, 4096)
        xyz = pts.transpose(1, 2).contiguous().cpu().numpy()
    kps, _, _, sal, rad = _iss(_cuda(xyz), rs, rnm, **kw)
    compared = ambiguous = 0
    for b in range(len(xyz)):
        c, a = _compare(xyz[b].T.copy(), kps[b], sal[b], rad[b], rs, rnm, **kw)
        compared += c; ambiguous += a
    share = ambiguous / (compared + ambiguous)
    print("%s: %d points compared, ambiguous share %.4f, keypoints %s" % (case, compared, share,
                                                                          [len(k) for k in kps]))
    assert share < 0.15
    assert sum(len(k) for k in kps) > 0


def test_returned_radii_reproduce_the_automatic_run():
    x = _cuda(_modelnet(8, 1024, seed=12))
    _, idx, cnt, sal, rad = _iss(x)
    for b in range(8):
        _, idx2, cnt2, sal2, rad2 = _iss(x[b:b + 1], float(rad[b, 0]), float(rad[b, 1]))
        assert np.array_equal(idx2[0], idx[b]) and cnt2[0] == cnt[b]
        assert np.array_equal(sal2[0].view(np.int64), sal[b].view(np.int64))
        assert np.array_equal(rad2[0], rad[b])


# ---------------------------------------------------------------------------------------------- 2. invariance
def test_rigid_motion_invariance():
    import ri_b200
    xyz = _modelnet(8, 1024, seed=13)
    rng = np.random.default_rng(13)
    R = ri_b200.synth.random_rotations(rng, 8)
    t = rng.uniform(-2, 2, (8, 3, 1))
    moved = (np.einsum('bij,bjn->bin', R, xyz.astype(np.float64)) + t).astype(np.float32)
    ka = _iss(_cuda(xyz))[0]
    kb = _iss(_cuda(moved))[0]
    total = excluded = 0
    for b in range(8):
        amb = O.iss(xyz[b].T.copy())['amb'] | O.iss(moved[b].T.copy())['amb']
        a = np.zeros(1024, bool); a[ka[b]] = True
        m = np.zeros(1024, bool); m[kb[b]] = True
        assert np.array_equal(a[~amb], m[~amb]), (b, int((a != m)[~amb].sum()))
        total += int(a[~amb].sum()); excluded += int(amb.sum())
    assert total > 50 and excluded < 0.25 * 8 * 1024


# ---------------------------------------------------------------------------------------------- 3. reproducibility
def test_bit_reproducible_and_batch_independent():
    xyz = np.concatenate([_modelnet(6, 2048, seed=14), _scans(2, 2048, seed=14)])
    x = _cuda(xyz)
    r1 = _iss(x)[1:]
    r2 = _iss(x)[1:]
    for a, b in zip(r1, r2):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    for b in (0, 3, 7):
        alone = _iss(x[b:b + 1])[1:]
        for a, full in zip(alone, r1):
            assert np.array_equal(a[0:1].view(np.uint8), full[b:b + 1].view(np.uint8))


# ---------------------------------------------------------------------------------------------- 4. degenerate inputs
def test_edge_cases():
    import torch
    import ri_b200
    F = ri_b200.functional.compute_iss_keypoints
    idx, cnt, sal, rad = F(torch.empty(0, 3, 100, device="cuda"), return_saliency=True, return_radii=True)
    assert idx.shape == (0, 100) and cnt.shape == (0,) and sal.shape == (0, 100) and rad.shape == (0, 2)
    idx, cnt, sal, rad = F(torch.empty(3, 3, 0, device="cuda"), return_saliency=True, return_radii=True)
    assert idx.shape == (3, 0) and cnt.tolist() == [0, 0, 0] and torch.all(rad == 0)
    idx, cnt, rad = F(torch.rand(2, 3, 1, device="cuda"), return_radii=True)
    assert cnt.tolist() == [0, 0] and idx.tolist() == [[-1], [-1]] and torch.all(rad == 0)
    idx, cnt = F(torch.rand(2, 3, 1, device="cuda"), 0.5, 0.5, min_neighbors=1)   # e3 of one point: C is zero
    assert cnt.tolist() == [0, 0]
    idx, cnt, sal, rad = F(torch.full((1, 3, 500), 0.3, device="cuda"), return_saliency=True, return_radii=True)
    assert int(cnt[0]) == 0 and torch.all(rad == 0) and torch.all(sal == 0) and torch.all(idx == -1)
    idx, cnt, sal = F(torch.full((1, 3, 500), 0.3, device="cuda"), 0.1, 0.1, return_saliency=True)
    assert int(cnt[0]) == 0 and torch.all(sal == 0)
    # NaN / inf points: never keypoints, never neighbours, not counted in the resolution
    X = _modelnet(1, 1024, seed=15)[0].T.copy()
    Y = X.copy()
    Y[[5, 77, 400]] = np.nan
    Y[600, 1] = np.inf
    kp, _, _, sal, rad = _iss(_cuda(Y.T[None]))
    assert not np.isin([5, 77, 400, 600], kp[0]).any() and np.all(sal[0, [5, 77, 400, 600]] == 0)
    _compare(Y, kp[0], sal[0], rad[0])
    # duplicates: equal saliency, both kept
    k = int(_iss(_cuda(X.T[None]))[0][0][0])
    D = np.concatenate([X, X[k:k + 1]])
    kp, _, _, sal, rad = _iss(_cuda(D.T[None]))
    assert k in kp[0] and 1024 in kp[0] and sal[0, k] == sal[0, 1024]
    _compare(D, kp[0], sal[0], rad[0])


# ---------------------------------------------------------------------------------------------- 5. argument errors
def test_argument_errors():
    import torch
    import ri_b200
    from ri_b200 import _lib
    x = torch.rand(2, 3, 256, device="cuda")
    op = torch.ops.ri.iss_keypoints
    bad = [(x.cpu(), 0., 0., .9, .9, 5), (x.double(), 0., 0., .9, .9, 5), (x[:, :2].contiguous(), 0., 0., .9, .9, 5),
           (x.transpose(1, 2), 0., 0., .9, .9, 5), (x, -0.1, 0.1, .9, .9, 5), (x, 0.1, float("nan"), .9, .9, 5),
           (x, float("inf"), 0.1, .9, .9, 5), (x, 0.1, 0.1, 0.0, .9, 5), (x, 0.1, 0.1, .9, float("nan"), 5),
           (x, 0.1, 0.1, .9, .9, 0), (torch.rand(65536, 3, 1, device="cuda"), 0., 0., .9, .9, 5)]
    for args in bad:
        with pytest.raises(RuntimeError):
            op(*args, False)
    with pytest.raises(RuntimeError):
        ri_b200.functional.compute_iss_keypoints(x, min_neighbors=0)
    idx = torch.empty(2, 256, dtype=torch.int32, device="cuda")
    cnt = torch.empty(2, dtype=torch.int32, device="cuda")
    nws = _lib.lib.ri_iss_workspace_bytes(2, 256)
    ws = torch.empty(nws + 256, dtype=torch.uint8, device="cuda")
    def call(rs=0.1, rnm=0.1, g21=0.9, g32=0.9, mn=5, i=idx.data_ptr(), c=cnt.data_ptr(), w=ws.data_ptr(), nb=nws, B=2,
             gamma=True):
        g = (ctypes.c_double * 2)(g21, g32) if gamma else None
        return _lib.lib.ri_iss_keypoints_f32(x.data_ptr(), B, 256, rs, rnm, g, mn, i, c, None, None, w, nb, None)
    assert call(rs=-1.0) == -1 and call(rnm=float("nan")) == -1 and call(rs=float("inf")) == -1
    assert call(g21=0.0) == -1 and call(g32=-1.0) == -1 and call(mn=0) == -1
    assert call(i=None) == -1 and call(c=None) == -1 and call(B=-1) == -1 and call(gamma=False) == -1
    assert call(B=65536) == -3
    assert call(nb=nws - 1) == -2 and call(w=None) == -2 and call(w=ws.data_ptr() + 16) == -2
    assert call() == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------- 6. the keypoint batch
def test_keypoint_batch_padding_leaves_matches_unchanged():
    import torch
    import ri_b200
    xyz = _modelnet(8, 1024, seed=16)
    x = _cuda(xyz)
    feats = torch.randn(8, 33, 1024, device="cuda")
    idx, cnt = ri_b200.functional.compute_iss_keypoints(x)
    pts, f, sel = ri_b200.functional.keypoint_batch(x, idx, cnt, feats)
    K = int(cnt.max())
    assert pts.shape == (8, K, 3) and f.shape == (8, K, 33) and sel.shape == (8, K) and int(cnt.min()) < K
    c = cnt.cpu().numpy()
    for b in range(8):
        kb = idx[b, :c[b]].long()
        assert torch.equal(sel[b, :c[b]].long(), kb) and torch.all(sel[b, c[b]:] == kb[0])
        assert torch.equal(pts[b, :c[b]], x[b, :, kb].T) and torch.equal(f[b, :c[b]], feats[b, :, kb].T)
    # pairs (b, b+1): padded batch against per-pair calls on exactly count[b] rows
    m = ri_b200.matcher.mutual_nn(f[0::2], f[1::2], point_major=True)
    for p in range(4):
        a, b = 2 * p, 2 * p + 1
        one = ri_b200.matcher.mutual_nn(f[a:a + 1, :c[a]].contiguous(), f[b:b + 1, :c[b]].contiguous(), point_major=True)
        k = int(one['count'][0])
        assert int(m['count'][p]) == k
        assert torch.equal(m['idx1'][p, :k], one['idx1'][0, :k]) and torch.equal(m['idx2'][p, :k], one['idx2'][0, :k])
    # a cloud with no keypoints is padded with its point 0
    flat = torch.zeros(1, 3, 64, device="cuda"); flat[0, :2] = torch.rand(2, 64, device="cuda")
    i0, c0 = ri_b200.functional.compute_iss_keypoints(flat)
    pts0, none, sel0 = ri_b200.functional.keypoint_batch(flat, i0, c0)
    assert int(c0[0]) == 0 and none is None and sel0.tolist() == [[0]] and torch.equal(pts0[0, 0], flat[0, :, 0])


# ---------------------------------------------------------------------------------------------- 7. the chain
def _terrain_pair(N, seed, jitter=0.001):
    """A bumpy height field and its copy under a random SE(3) plus independent jitter, xyz only.
    -> (src [N,3], tgt [N,3], G [4,4] src -> tgt, camera above the source, the same camera in the target frame)."""
    import ri_b200
    rng = np.random.default_rng(seed)
    uv = rng.uniform(-1, 1, (N, 2))
    z = np.zeros(N)
    for _ in range(8):
        c = rng.uniform(-1, 1, 2); s = rng.uniform(0.15, 0.4); a = rng.uniform(-0.4, 0.4)
        z += a * np.exp(-np.sum((uv - c) ** 2, 1) / (2 * s * s))
    src = np.column_stack([uv, z])
    G = np.eye(4)
    G[:3, :3] = ri_b200.synth.random_rotations(rng, 1)[0]
    G[:3, 3] = rng.uniform(-0.5, 0.5, 3)
    tgt = src @ G[:3, :3].T + G[:3, 3] + rng.standard_normal(src.shape) * jitter
    cam = np.array([0.0, 0.0, 5.0])
    return src.astype(np.float32), tgt.astype(np.float32), G, cam, G[:3, :3] @ cam + G[:3, 3]


def test_registration_chain_on_keypoints():
    import torch
    import ri_b200
    from scipy.spatial import cKDTree
    P, N, r_n, r_f, voxel = 3, 2048, 0.1, 0.3, 0.05
    pairs = [_terrain_pair(N, 100 + s) for s in range(P)]
    src = np.stack([p[0] for p in pairs]); tgt = np.stack([p[1] for p in pairs])
    s_cm, t_cm = _cuda(src.transpose(0, 2, 1)), _cuda(tgt.transpose(0, 2, 1))
    cam_s = torch.tensor(np.stack([p[3] for p in pairs]), dtype=torch.float32, device="cuda")
    cam_t = torch.tensor(np.stack([p[4] for p in pairs]), dtype=torch.float32, device="cuda")
    F = ri_b200.functional
    fs = F.compute_fpfh_feature(s_cm, F.estimate_normals(s_cm, r_n, 30, camera=cam_s), r_f, 100)
    ft = F.compute_fpfh_feature(t_cm, F.estimate_normals(t_cm, r_n, 30, camera=cam_t), r_f, 100)
    ks, cs, rad_s = F.compute_iss_keypoints(s_cm, return_radii=True)
    kt, ct = F.compute_iss_keypoints(t_cm)
    # repeatability under the ground truth: share of source keypoints with a target keypoint within r_nm.  The oracle gives
    # 0.77 / 0.83 / 0.91 on these three pairs (tests/iss_oracle.py on the CPU); 0.6 leaves room for ambiguous points.
    for p in range(P):
        G = pairs[p][2]
        a = src[p][ks[p, :cs[p]].cpu().numpy()] @ G[:3, :3].T + G[:3, 3]
        d, _ = cKDTree(tgt[p][kt[p, :ct[p]].cpu().numpy()]).query(a)
        rep = float(np.mean(d < float(rad_s[p, 1])))
        assert rep >= 0.6, (p, rep)
    ps, fks, _ = F.keypoint_batch(s_cm, ks, cs, fs)
    pt, fkt, _ = F.keypoint_batch(t_cm, kt, ct, ft)
    m = ri_b200.matcher.mutual_nn(fks, fkt, point_major=True, want_dist=False)
    s_pm, t_pm = _cuda(src), _cuda(tgt)
    extent = max(np.linalg.norm(src[p].max(0) - src[p].min(0)) for p in range(P))
    for func in ('ransac', 'fgr'):
        T, _ = ri_b200.registration.estimate_poses(ps, pt, m['idx1'], m['idx2'], m['count'], func=func, voxel_size=voxel)
        T = ri_b200.registration.icp(s_pm, t_pm, 2 * voxel, init=T)['transformation'].cpu().numpy()
        for p in range(P):
            G = pairs[p][2]
            D = T[p][:3, :3].astype(np.float64) @ G[:3, :3].T
            rre = math.degrees(math.acos(min(1.0, max(-1.0, (np.trace(D) - 1) / 2))))
            rte = float(np.linalg.norm(T[p][:3, 3] - G[:3, 3]))
            assert rre < 1.0 and rte < 0.01 * extent, (func, p, rre, rte, int(m['count'][p]))
