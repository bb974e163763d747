"""Row f10 on the GPU: csrc/teaser.cu against its fp64 replay (tests/teaser_oracle.py).

The clique (its size, the exact flag and the ascending match positions) must equal the replay's exactly: the graph is
built from bit-exact edge lengths and the search order is fixed.  The pose must be the replay's to 1e-5 on fixtures the
replay shows to be well conditioned (a clear eigen gap in every Horn step, no residual near a weight threshold), and the
inlier count must agree with a recount under the returned pose.  Then: ground truth at high outlier rates, degenerate
pairs, coordinates far from the origin, determinism, pair independence, the estimate_poses / meter wiring and argument
errors.
"""
import numpy as np
import pytest

import pose_oracle as po
import teaser_oracle as to
from test_pose_gpu import batch, matched

NB = 0.03                      # noise bound of the planted fixtures (5 mm noise per axis)


def teaser_call(src, tgt, idx1, idx2, count, noise_bound=NB, cbar2=1.0, gnc_factor=1.4, max_iterations=100,
                cost_threshold=1e-12, max_clique_nodes=1 << 20, inlier_dist=NB):
    import torch
    import ri_b200  # noqa: F401
    d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (src, tgt, idx1, idx2, count)]
    out = torch.ops.ri.teaser(*d, noise_bound, cbar2, gnc_factor, max_iterations, cost_threshold, max_clique_nodes,
                              inlier_dist)
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in out]


def check(data, pose=True, tol_t=1e-5, **kw):
    """The kernels against the replay on every pair of `data`; -> (GPU outputs, replays)."""
    rkw = dict(kw)                                      # the replay takes the op's option names
    rkw.setdefault("noise_bound", NB)
    rkw.setdefault("inlier_dist", NB)
    want = [to.replay(*matched(*data, p), **rkw) for p in range(len(data[4]))]
    T, inl, clique, size, exact = got = teaser_call(*data, **kw)
    for p, r in enumerate(want):
        K = len(r.clique)
        assert size[p] == K and bool(exact[p]) == r.exact, (p, size[p], K, exact[p], r.exact)
        assert np.array_equal(clique[p, :K], r.clique) and np.all(clique[p, K:] == -1), p
        if not r.posed:
            assert np.array_equal(T[p], np.eye(4, dtype=np.float32)) and inl[p] == 0, p
            continue
        if pose:
            g = r.gnc                                   # max_iterations = 0: no Horn step, R = I on both sides
            assert min(g.gaps, default=1.0) > 1e-6 * max(1.0, K) and min(g.margins, default=1.0) > 1e-6, \
                ("ill-conditioned fixture", p)
            assert np.abs(T[p, :3, :3] - r.T[:3, :3]).max() < 1e-5, (p, T[p], r.T)
            assert np.abs(T[p, :3, 3] - r.T[:3, 3]).max() < tol_t, (p, T[p], r.T)
        assert np.array_equal(T[p, 3], [0, 0, 0, 1])
        a, b = matched(*data, p)
        assert abs(int(inl[p]) - to.count_inliers(T[p], a, b, rkw["inlier_dist"])) <= 2, p
    return got, want


def planted(counts, outliers, seed, n=None, offset=0.0):
    rng = np.random.default_rng(seed)
    outl = outliers if isinstance(outliers, (list, tuple)) else [outliers] * len(counts)
    pairs = [po.planted_matches(rng, m, o, offset=offset) for m, o in zip(counts, outl)]
    return batch([x[:2] for x in pairs], n=n, seed=seed), [x[2] for x in pairs]


RAGGED = [700, 1000, 333, 1024, 517]


# ---------------------------------------------------------------------------------------------- the clique, exactly
@pytest.mark.gpu
@pytest.mark.parametrize("outliers", [0.0, 0.5, 0.9, 0.99])
def test_clique_and_pose_outliers(outliers):
    data, _ = planted(RAGGED, outliers, seed=int(outliers * 100) + 1, n=1100)
    check(data, pose=outliers < 0.99)


@pytest.mark.gpu
@pytest.mark.parametrize("noise_bound", [0.015, 0.03, 0.1])
def test_noise_bounds(noise_bound):
    data, _ = planted(RAGGED, 0.5, seed=3, n=1100)
    check(data, noise_bound=noise_bound, inlier_dist=noise_bound, pose=False)


@pytest.mark.gpu
@pytest.mark.parametrize("m", [3, 1023, 1024, 1025, 4097])
def test_match_counts(m):
    rng = np.random.default_rng(m)
    a, b, _, _ = po.planted_matches(rng, m, 0.5 if m > 3 else 0.0)
    other = po.planted_matches(rng, 600, 0.5)[:2]
    check(batch([other, (a, b)], n=max(m, 600), seed=m), pose=m > 3)


@pytest.mark.gpu
def test_scan_sized_pair():
    # ~20k matches of one pair: 625 words per bitset row
    data, _ = planted([20011], 0.9, seed=20, n=20011)
    check(data, pose=False)


@pytest.mark.gpu
def test_budget_exhausted_gives_partial_clique():
    # a dense random graph (all outliers, generous bound) with a budget of a few nodes: exact = 0 and the replay's
    # partial clique bit for bit
    data, _ = planted([300, 200], 1.0, seed=30, n=300)
    full = [to.replay(*matched(*data, p), noise_bound=0.2).search for p in range(2)]
    assert all(f.exact and f.nodes > 3 for f in full)
    (_, _, _, _, exact), want = check(data, noise_bound=0.2, inlier_dist=0.2, max_clique_nodes=3, pose=False)
    assert not exact.any() and not any(w.exact for w in want)


# ---------------------------------------------------------------------------------------------- options, ground truth
@pytest.mark.gpu
@pytest.mark.parametrize("gnc_factor,max_iterations", [(1.4, 100), (2.0, 100), (1.4, 1), (1.4, 0)])
def test_gnc_options(gnc_factor, max_iterations):
    data, _ = planted(RAGGED, 0.5, seed=40, n=1100)
    check(data, gnc_factor=gnc_factor, max_iterations=max_iterations)


@pytest.mark.gpu
def test_recovers_ground_truth_at_95_percent_outliers():
    data, gts = planted([1000, 2000, 1024], 0.95, seed=95, n=2000)
    (T, inl, _, _, _), _ = check(data, pose=False)
    for p, gt in enumerate(gts):
        R = T[p, :3, :3].astype(np.float64) @ gt[:3, :3].T
        assert np.degrees(np.arccos(np.clip((np.trace(R) - 1) / 2, -1, 1))) < 1.0, p
        assert np.linalg.norm(T[p, :3, 3] - gt[:3, 3]) < 0.02, p


@pytest.mark.gpu
def test_far_from_origin():
    data, _ = planted([800, 1000, 611], 0.5, seed=60, n=1000, offset=100.0)
    check(data, tol_t=1e-5 * 101)


# ---------------------------------------------------------------------------------------------- degenerate, batch
@pytest.mark.gpu
def test_degenerate_pairs_in_one_batch():
    rng = np.random.default_rng(41)
    good = [po.planted_matches(rng, 500, 0.5)[:2] for _ in range(2)]
    a3 = np.array([[0, 0, 0], [1, 0, 0], [0, 2, 0]], np.float32)
    b3 = np.array([[0, 0, 0], [3, 0, 0], [0, 7, 0]], np.float32)
    pairs = [good[0], (a3[:0], b3[:0]), (a3[:2], b3[:2]), (a3, b3), good[1]]
    data = batch(pairs, n=600, seed=42)
    (T, inl, _, size, _), want = check(data, pose=False)
    eye = np.eye(4, dtype=np.float32)
    for p in (1, 2, 3):
        assert np.array_equal(T[p], eye) and inl[p] == 0 and size[p] < 3, p
    assert want[0].posed and want[4].posed


@pytest.mark.gpu
def test_deterministic_and_pairs_independent():
    rng = np.random.default_rng(70)
    pairs = [po.planted_matches(rng, m, 0.6)[:2] for m in (900, 3000, 77)]
    data = batch(pairs, n=3000, seed=71)
    r1 = teaser_call(*data)
    r2 = teaser_call(*data)
    assert all(np.array_equal(x, y) for x, y in zip(r1, r2))
    for p in range(3):
        other = [x.copy() for x in data]
        src, tgt, idx1, idx2, count = other
        q = [i for i in range(3) if i != p]
        src[q] = rng.uniform(-1, 1, src[q].shape); tgt[q] = rng.uniform(-1, 1, tgt[q].shape)
        idx1[q] = rng.integers(0, 3000, idx1[q].shape); count[q] = rng.integers(0, 3000, len(q))
        r3 = teaser_call(*other)
        assert all(np.array_equal(x[p], y[p]) for x, y in zip(r3, r1)), p
    alone = teaser_call(*(x[:1] for x in data))
    assert all(np.array_equal(x[0], y[0]) for x, y in zip(alone, r1))


# ---------------------------------------------------------------------------------------------- public interface
@pytest.mark.gpu
def test_estimate_poses_mapping():
    import torch
    import ri_b200
    data, _ = planted(RAGGED, 0.5, seed=12, n=1100)
    d = [torch.from_numpy(x).cuda() for x in data]
    with pytest.raises(ValueError, match="noise_bound"):
        ri_b200.registration.estimate_poses(*d, func='teaserpp')
    T, inl = ri_b200.registration.estimate_poses(*d, func='teaserpp', voxel_size=0.08, noise_bound=NB, seed=5)
    r = ri_b200.registration.teaser(*d, NB, inlier_dist=0.08, return_clique=True)
    assert torch.equal(T, r['transformation']) and torch.equal(inl, r['inliers'])
    assert r['clique_exact'].dtype == torch.bool and bool(r['clique_exact'].all())
    assert torch.equal((r['clique'] >= 0).sum(1).int(), r['clique_size'])
    # the other modes ignore noise_bound
    T1, _ = ri_b200.registration.estimate_poses(*d, func='kabsch', noise_bound=NB)
    T2, _ = ri_b200.registration.estimate_poses(*d, func='kabsch')
    assert torch.equal(T1, T2)


@pytest.mark.gpu
@pytest.mark.parametrize("icp", [None, {'max_correspondence_distance': 0.05}])
def test_meter_end_to_end(icp):
    import ri_b200
    rng = np.random.default_rng(5)
    P, n, C = 4, 512, 64
    src = rng.uniform(-1, 1, (P, n, 3)).astype(np.float32)
    gt = np.stack([po.rand_pose(rng) for _ in range(P)]).astype(np.float32)
    desc = rng.standard_normal((P, C, n)).astype(np.float32)
    perm = np.stack([rng.permutation(n) for _ in range(P)])
    tgt = np.empty_like(src); desc2 = np.empty_like(desc)
    for p in range(P):
        tgt[p, perm[p]] = src[p] @ gt[p, :3, :3].T + gt[p, :3, 3]
        desc2[p][:, perm[p]] = desc[p] + 0.01 * rng.standard_normal((C, n)).astype(np.float32)
    with pytest.raises(ValueError, match="noise_bound"):
        ri_b200.registration.MeterModelNet40_registration('teaserpp', icp=icp)
    meter = ri_b200.registration.MeterModelNet40_registration('teaserpp', icp=icp, noise_bound=0.01)
    meter.update((desc, desc2), (src, tgt, gt))
    r = meter.compute()
    assert set(r) == {'succ', 'rre', 'rte', 'rmse', 'reg_time', 'rmse_succ'}
    assert r['rmse_succ'] == 1.0 and r['rre'] < 0.05 and r['rte'] < 1e-3 and r['rmse'] < 1e-3, r


@pytest.mark.gpu
def test_argument_errors():
    import torch
    import ri_b200  # noqa: F401
    P, n = 3, 40
    f = lambda *s: torch.rand(*s, device="cuda")
    i = lambda *s: torch.zeros(*s, dtype=torch.int32, device="cuda")
    ok = dict(src=f(P, n, 3), tgt=f(P, n + 5, 3), idx1=i(P, n), idx2=i(P, n), count=i(P))
    opts = dict(noise_bound=0.01, cbar2=1.0, gnc_factor=1.4, max_iterations=100, cost_threshold=1e-12,
                max_clique_nodes=1000, inlier_dist=0.01)
    op = torch.ops.ri.teaser
    call = lambda kw, **o: op(kw["src"], kw["tgt"], kw["idx1"], kw["idx2"], kw["count"], *{**opts, **o}.values())
    call(ok)
    bad = [dict(src=f(P, n)), dict(src=f(P, n, 4)), dict(tgt=f(P, n, 2)), dict(tgt=f(P + 1, n, 3)),
           dict(idx1=i(P, n + 1)), dict(idx2=i(P, n - 1)), dict(count=i(P, 1)), dict(count=i(P + 1)),
           dict(src=f(P, n, 3).cpu()), dict(idx1=i(P, n).long())]
    for b in bad:
        with pytest.raises(RuntimeError):
            call({**ok, **b})
    inf = float("inf")
    for o in (dict(noise_bound=0.0), dict(noise_bound=-1.0), dict(noise_bound=inf), dict(noise_bound=float("nan")),
              dict(cbar2=0.0), dict(cbar2=inf), dict(inlier_dist=0.0), dict(inlier_dist=inf), dict(gnc_factor=1.0),
              dict(max_iterations=-1), dict(max_clique_nodes=0)):
        with pytest.raises(RuntimeError):
            call(ok, **o)
    big = dict(ok, idx1=i(1, (1 << 15) + 1), idx2=i(1, (1 << 15) + 1), src=f(1, n, 3), tgt=f(1, n, 3), count=i(1))
    with pytest.raises(RuntimeError, match="unsupported"):
        call(big)
    torch.cuda.synchronize()
