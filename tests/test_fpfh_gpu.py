"""Row f8 (SURVEY.md §8f): batched FPFH descriptors on the GPU (csrc/fpfh.cu) against the k-NN their neighbour lists are
defined by and the numpy reference (tests/fpfh_oracle.py) on those lists, degenerate inputs, reproducibility, argument
errors, and the xyz-only registration chain estimate_normals -> compute_fpfh_feature -> mutual_nn -> pose -> ICP."""

import numpy as np
import pytest

import fpfh_oracle as ref

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- helpers
def _modelnet(B, N, seed):
    import ri_b200
    c = ri_b200.synth.make_clouds(B, N, seed=seed)
    return np.ascontiguousarray(c[:, :3]), np.ascontiguousarray(c[:, 3:])


def _cuda(*arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


def _lim(r):
    r = np.float32(r)
    return float(min(r * r, np.float32(10000.0)))


def _fpfh(x, n, r, max_nn):
    """-> (fpfh, counts, bin counts recovered from spfh) as numpy."""
    import ri_b200
    f, cnt, sp = ri_b200.functional.compute_fpfh_feature(x, n, r, max_nn, return_counts=True, return_spfh=True)
    cnt = cnt.cpu().numpy()
    sp = sp.cpu().numpy().astype(np.float64)
    c = np.rint(sp * np.maximum(cnt - 1, 0)[:, None, :] / 100.0).astype(np.int64)
    return f.cpu().numpy(), cnt, c


def _knn_lists(x, r, max_nn):
    """The k-NN's lists cut at the radius: (idx [B,N,max_nn], count [B,N]) as numpy."""
    import ri_b200
    dist, idx = ri_b200.functional.knn_indices(x, max_nn)
    cnt = (dist < _lim(r)).sum(1).int()
    return idx.cpu().numpy().transpose(0, 2, 1), cnt.cpu().numpy()


def _against_oracle(xyz, nrm, r, max_nn, check_values=True):
    """GPU counts, bin counts and FPFH vs the oracle on the k-NN's lists; -> (points compared, ambiguous points)."""
    x, n = _cuda(xyz, nrm)
    f, cnt, c = _fpfh(x, n, r, max_nn)
    idx, want = _knn_lists(x, r, max_nn)
    assert np.array_equal(cnt, want), (max_nn, r, int((cnt != want).sum()))
    compared = ambiguous = 0
    for b in range(len(xyz)):
        p, q = xyz[b].T, nrm[b].T
        of, osp, oc, amb = ref.compute_fpfh(p, q, idx[b], cnt[b])
        gc = c[b].T
        assert np.array_equal(gc[~amb], oc[~amb]), (b, int((gc[~amb] != oc[~amb]).any(1).sum()))
        ambiguous += int(amb.sum())
        if check_values:
            nb_amb = np.array([amb[idx[b, i, :cnt[b, i]]].any() for i in range(len(p))])
            ok = ~amb & ~nb_amb
            g = f[b].T.astype(np.float64)
            scale = np.repeat(np.abs(of).reshape(-1, 3, 11).max(2), 11, axis=1)
            err = np.abs(g - of)[ok] / np.maximum(scale[ok], 1e-30)
            assert err.max(initial=0.0) <= 1e-6, (b, err.max())
            compared += int(ok.sum())
    return compared, ambiguous


# ---------------------------------------------------------------------------------------------- 1. lists and counts
@pytest.mark.parametrize("max_nn", [1, 2, 31, 32, 33, 64, 100, 128])
def test_counts_and_bins_equal_knn_lists(max_nn):
    xyz, nrm = _modelnet(4, 1024, seed=1)
    for r in (0.05, 0.25, float("inf")):
        _, amb = _against_oracle(xyz, nrm, r, max_nn, check_values=False)
        assert amb < 0.01 * xyz.shape[0] * xyz.shape[2], (max_nn, r, amb)


# ---------------------------------------------------------------------------------------------- 2. values
@pytest.mark.parametrize("max_nn,r", [(100, 0.25), (128, 0.4), (33, float("inf"))])
def test_fpfh_values_match_oracle(max_nn, r):
    xyz, nrm = _modelnet(8, 1024, seed=2)
    compared, amb = _against_oracle(xyz, nrm, r, max_nn)
    total = xyz.shape[0] * xyz.shape[2]
    print("fpfh max_nn=%d r=%s: %d ambiguous points of %d, %d values compared" % (max_nn, r, amb, total, compared))
    assert amb < 0.01 * total and compared > 0.5 * total, (amb, compared)


def test_dense_cluster_many_compactions():
    """Thousands of points inside one radius: the per-warp key buffer is compacted many times per query."""
    rng = np.random.default_rng(3)
    ball = rng.standard_normal((4000, 3)) * 0.01
    rest = rng.uniform(-1, 1, (2000, 3))
    p = np.concatenate([ball, rest])[rng.permutation(6000)]
    nrm = rng.standard_normal((6000, 3)); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    xyz = p.T[None].astype(np.float32); nn = nrm.T[None].astype(np.float32)
    for max_nn in (100, 128):
        _, amb = _against_oracle(xyz, nn, 0.1, max_nn)
        assert amb < 60, amb


# ---------------------------------------------------------------------------------------------- 3. degenerate inputs
def test_degenerate_inputs():
    import torch
    rng = np.random.default_rng(4)
    # exact duplicates, several copies each, shuffled so q is often not at list position 0
    base = rng.uniform(-1, 1, (300, 3))
    p = np.concatenate([base, base[:100], base[:50]])[rng.permutation(450)]
    nrm = rng.standard_normal((450, 3)); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    xyz = p.T[None].astype(np.float32); nn = nrm.T[None].astype(np.float32)
    _against_oracle(xyz, nn, 0.3, 40)
    x, n = _cuda(xyz, nn)
    idx, cnt = _knn_lists(x, 0.3, 40)
    assert (idx[0, :, 0] != np.arange(450)).any()                        # some q sorts behind its duplicate
    # zero normals: every pair feature is (0,0,0), so all counts sit in bins 5, 16, 27
    f, c_, c = _fpfh(x, torch.zeros_like(n), 0.3, 40)
    many = c_[0] > 1
    assert (c[0, [5, 16, 27]][:, many] == c_[0][many] - 1).all() and c[0].sum() == 3 * (c_[0][many] - 1).sum()
    _against_oracle(xyz, np.zeros_like(nn), 0.3, 40)
    # isolated points: n = 1, zeros
    grid = np.stack(np.meshgrid(np.arange(6), np.arange(6), np.arange(6)), 0).reshape(1, 3, -1).astype(np.float32)
    g, = _cuda(grid)
    f, cnt, c = _fpfh(g, g, 0.5, 30)
    assert (cnt == 1).all() and (f == 0).all() and (c == 0).all()
    # N = 1 and max_nn > N
    f, cnt, _ = _fpfh(*_cuda(xyz[:, :, :1], nn[:, :, :1]), 1.0, 10)
    assert (cnt == 1).all() and (f == 0).all()
    _against_oracle(xyz[:, :, :10].copy(), nn[:, :, :10].copy(), float("inf"), 50)
    # empty batches
    for shape in ((0, 3, 100), (3, 3, 0)):
        e = torch.empty(shape, device="cuda")
        import ri_b200
        assert tuple(ri_b200.functional.compute_fpfh_feature(e, e, 0.1).shape) == (shape[0], 33, shape[2])


# ---------------------------------------------------------------------------------------------- 4. invariance
def test_rigid_invariance():
    import ri_b200
    xyz, nrm = _modelnet(4, 1024, seed=5)
    R = ri_b200.synth.random_rotations(np.random.default_rng(6), 4)
    xyz2 = (np.einsum('bij,bjn->bin', R, xyz) + np.array([0.3, -0.2, 0.1])[None, :, None]).astype(np.float32)
    nrm2 = np.einsum('bij,bjn->bin', R, nrm).astype(np.float32)
    r, k = 0.25, 100
    a = _fpfh(*_cuda(xyz, nrm), r, k)
    b = _fpfh(*_cuda(xyz2, nrm2), r, k)
    la, _ = _knn_lists(_cuda(xyz)[0], r, k)
    lb, _ = _knn_lists(_cuda(xyz2)[0], r, k)
    checked = 0
    for c in range(4):
        # points whose list is the same on both copies and whose bins are clear of an edge by 1e-5 on both
        same = (a[1][c] == b[1][c]) & np.array([np.array_equal(la[c, i, :a[1][c, i]], lb[c, i, :a[1][c, i]])
                                                for i in range(1024)])
        _, am1 = ref.spfh_counts(xyz[c].T, nrm[c].T, la[c], a[1][c], bin_tol=1e-5, swap_tol=1e-5)
        _, am2 = ref.spfh_counts(xyz2[c].T, nrm2[c].T, lb[c], b[1][c], bin_tol=1e-5, swap_tol=1e-5)
        ok = same & ~am1 & ~am2
        assert ok.mean() > 0.9, ok.mean()
        assert np.array_equal(a[2][c][:, ok], b[2][c][:, ok])
        nb = ok & np.array([ok[la[c, i, :a[1][c, i]]].all() for i in range(1024)])
        fa, fb = a[0][c][:, nb].astype(np.float64), b[0][c][:, nb].astype(np.float64)
        assert np.abs(fa - fb).max() <= 1e-4 * np.abs(fa).max()
        checked += int(nb.sum())
    assert checked > 0.1 * 4 * 1024, checked


# ---------------------------------------------------------------------------------------------- 5. reproducibility
def test_deterministic_and_clouds_independent():
    import torch
    import ri_b200
    xyz, nrm = _modelnet(5, 1024, seed=7)
    x, n = _cuda(xyz, nrm)
    run = lambda xx, nn: ri_b200.functional.compute_fpfh_feature(xx, nn, 0.25, 100)
    a, b = run(x, n), run(x, n)
    assert torch.equal(a, b)
    for c in range(5):
        assert torch.equal(run(x[c:c + 1], n[c:c + 1])[0], a[c]), c


# ---------------------------------------------------------------------------------------------- 6. argument errors
def test_errors():
    import torch
    import ri_b200
    from ri_b200 import _lib
    fn = ri_b200.functional.compute_fpfh_feature
    x = torch.rand(2, 3, 256, device="cuda")
    for bad in (dict(max_nn=0), dict(max_nn=129), dict(radius=0.0), dict(radius=-1.0), dict(radius=float("nan"))):
        kw = dict(radius=0.1, max_nn=30); kw.update(bad)
        with pytest.raises(RuntimeError):
            fn(x, x, kw.pop("radius"), **kw)
    for xx, nn in ((x.cpu(), x.cpu()), (x, x.cpu()), (x, x[:1].contiguous()), (x, x[:, :, :100].contiguous()),
                   (torch.rand(2, 4, 256, device="cuda"), torch.rand(2, 4, 256, device="cuda"))):
        with pytest.raises(RuntimeError):
            fn(xx, nn, 0.1)
    with pytest.raises(RuntimeError):
        torch.ops.ri.compute_fpfh(x.int(), x, 0.1, 30, False, False)
    out = torch.empty(2, 33, 256, device="cuda")
    ws = torch.empty(_lib.lib.ri_fpfh_workspace_bytes(2, 256, 128), dtype=torch.uint8, device="cuda")
    call = lambda r, k, nb=ws.numel(): _lib.lib.ri_compute_fpfh_f32(x.data_ptr(), x.data_ptr(), 2, 256, r, k,
                                                                    out.data_ptr(), None, None, ws.data_ptr(), nb, None)
    assert call(0.1, 129) == -3 and call(0.1, 0) == -1 and call(0.0, 30) == -1 and call(float("nan"), 30) == -1
    assert call(0.1, 128, 16) == -2
    assert call(0.1, 128) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------- 7. xyz-only registration
def _terrain_pair(N, seed, jitter=0.001):
    """A bumpy height field (distinctive local shape) and its copy under a random SE(3) plus independent jitter, xyz only.
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


def _rre_rte(T, G):
    D = np.asarray(T, np.float64)[:3, :3] @ G[:3, :3].T
    rre = np.degrees(np.arccos(np.clip((np.trace(D) - 1) / 2, -1, 1)))
    return rre, np.linalg.norm(np.asarray(T, np.float64)[:3, 3] - G[:3, 3])


def test_xyz_only_registration_chain():
    import torch
    import ri_b200
    from oracle import cpu_oracle
    P, N, r_n, r_f, voxel = 3, 2048, 0.1, 0.3, 0.05
    pairs = [_terrain_pair(N, 100 + s) for s in range(P)]
    src = np.stack([p[0] for p in pairs]); tgt = np.stack([p[1] for p in pairs])
    s_cm, t_cm = _cuda(src.transpose(0, 2, 1), tgt.transpose(0, 2, 1))
    cam_s = torch.tensor(np.stack([p[3] for p in pairs]), dtype=torch.float32, device="cuda")
    cam_t = torch.tensor(np.stack([p[4] for p in pairs]), dtype=torch.float32, device="cuda")
    ns = ri_b200.functional.estimate_normals(s_cm, r_n, 30, camera=cam_s)
    nt = ri_b200.functional.estimate_normals(t_cm, r_n, 30, camera=cam_t)
    fs = ri_b200.functional.compute_fpfh_feature(s_cm, ns, r_f, 100)
    ft = ri_b200.functional.compute_fpfh_feature(t_cm, nt, r_f, 100)
    m = ri_b200.matcher.mutual_nn(fs, ft, want_dist=False)
    fs_np, ft_np = fs.cpu().numpy(), ft.cpu().numpy()
    ns_np, nt_np = ns.cpu().numpy(), nt.cpu().numpy()
    is_, cs_ = _knn_lists(s_cm, r_f, 100)
    it_, ct_ = _knn_lists(t_cm, r_f, 100)
    for p in range(P):
        G = pairs[p][2]
        # registrable on the CPU: oracle FPFH on the same normals and lists, numpy mutual NN, ground-truth inlier ratio
        of_s = ref.compute_fpfh(src[p], ns_np[p].T, is_[p], cs_[p])[0].astype(np.float32)
        of_t = ref.compute_fpfh(tgt[p], nt_np[p].T, it_[p], ct_[p])[0].astype(np.float32)
        i1, i2, _ = cpu_oracle.find_correspondence_one_pair(of_s, of_t)
        gt = src[p][i1] @ G[:3, :3].T + G[:3, 3]
        ratio = np.mean(np.linalg.norm(gt - tgt[p][i2], axis=1) < voxel)
        assert ratio >= 0.3, (p, len(i1), ratio)
        # the GPU matches on the GPU descriptors against the reference method's on the same descriptors, with the parity
        # statement of test_matcher_gpu.py: every pick is an fp64 minimiser up to 1e-5 of the cancelling terms, and the
        # picks (and so the mutual matches) are equal wherever the reference's own fp32 matrix separates the minimum by 4x
        # that.  Smooth surfaces give many FPFH near-ties (a third of the rows here), so the separated share is only
        # required to be a majority, which keeps the equality check from being vacuous.
        a, b = fs_np[p].T.copy(), ft_np[p].T.copy()
        j1, j2, diff = cpu_oracle.find_correspondence_one_pair(a, b)
        x, y = a.astype(np.float64), b.astype(np.float64)
        d = (x * x).sum(1)[:, None] + (y * y).sum(1)[None, :] - 2 * x @ y.T
        tol = 1e-5 * ((x * x).sum(1).max() + (y * y).sum(1).max())
        c12, c21 = m['corr12'][p].cpu().numpy(), m['corr21'][p].cpu().numpy()
        assert (d[np.arange(len(a)), c12] - d.min(1)).max() <= tol and (d[c21, np.arange(len(b))] - d.min(0)).max() <= tol
        srt = np.sort(diff, 1); rows = srt[:, 1] - srt[:, 0] > 4 * tol
        srt = np.sort(diff, 0); cols = srt[1] - srt[0] > 4 * tol
        assert rows.mean() > 0.5 and cols.mean() > 0.5, (rows.mean(), cols.mean())
        o12, o21 = diff.argmin(1), diff.argmin(0)
        assert np.array_equal(c12[rows], o12[rows]) and np.array_equal(c21[cols], o21[cols])
        k = int(m['count'][p])
        mine = np.zeros(len(a), bool); mine[m['idx1'][p, :k].cpu().numpy()] = True
        theirs = np.zeros(len(a), bool); theirs[j1] = True
        sure = rows & cols[o12]                     # row i and the column it picks are both separated
        assert np.array_equal(mine[sure], theirs[sure]), int((mine[sure] != theirs[sure]).sum())
        assert np.array_equal(c12[mine], m['idx2'][p, :k].cpu().numpy())
    s_pm, t_pm = _cuda(src, tgt)
    extent = max(np.linalg.norm(src[p].max(0) - src[p].min(0)) for p in range(P))
    for func in ('ransac', 'fgr'):
        T, _ = ri_b200.registration.estimate_poses(s_pm, t_pm, m['idx1'], m['idx2'], m['count'], func=func,
                                                   voxel_size=voxel)
        T = ri_b200.registration.icp(s_pm, t_pm, 2 * voxel, init=T)['transformation'].cpu().numpy()
        for p in range(P):
            rre, rte = _rre_rte(T[p], pairs[p][2])
            assert rre < 1.0 and rte < 0.01 * extent, (func, p, rre, rte)
