"""Row f7 on the GPU: csrc/fgr.cu against its fp64 replay (tests/fgr_oracle.py).

The tuple list (corr, ncorr) must equal the replay's exactly: the sampler and the edge test are pinned bit for bit.  The
pose must be the replay's to 1e-5 on fixtures the replay shows to be well conditioned (every step solved, smallest
eigenvalue of J^T W J above 1), and the inlier count must agree with a recount under the returned pose.  Then: match counts
around and beyond the shared-memory staging of the list, ragged and degenerate pairs, coordinates far from the origin,
determinism, pair independence, the estimate_poses / meter wiring and argument errors.
"""
import numpy as np
import pytest

import fgr_oracle as fo
import pose_oracle as po
from test_pose_gpu import batch, matched

STAGE = 3072                    # list entries staged in shared memory


def fgr_call(src, tgt, idx1, idx2, count, max_corr_dist=0.025, iterations=64, division_factor=1.4,
             use_absolute_scale=False, decrease_mu=True, tuple_test=True, tuple_scale=0.95, max_tuples=1000, seed=0,
             inlier_dist=0.025):
    import torch
    import ri_b200  # noqa: F401
    d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (src, tgt, idx1, idx2, count)]
    seed = seed - (1 << 64) if seed >= 1 << 63 else seed                # the op takes the 64 bits as a signed int
    out = torch.ops.ri.fgr(*d, max_corr_dist, iterations, division_factor, use_absolute_scale, decrease_mu, tuple_test,
                           tuple_scale, max_tuples, seed, inlier_dist)
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in out]


def replays(src, tgt, idx1, idx2, count, **kw):
    return [fo.replay(src[p], tgt[p], *matched(src, tgt, idx1, idx2, count, p), pair=p, **kw) for p in range(len(count))]


def check(data, tol_t=1e-5, pose=True, **kw):
    """The kernel against the replay on every pair of `data`; -> (GPU outputs, replays)."""
    want = replays(*data, **kw)
    T, inl, corr, ncorr = got = fgr_call(*data, **kw)
    tuple_test = kw.get("tuple_test", True)
    for p, r in enumerate(want):
        assert ncorr[p] == len(r.corr), (p, ncorr[p], len(r.corr))
        if tuple_test:
            assert np.array_equal(corr[p, :ncorr[p]], r.corr), p
            assert np.all(corr[p, ncorr[p]:] == -1), p
        if not r.posed:
            assert np.array_equal(T[p], np.eye(4, dtype=np.float32)) and inl[p] == 0, p
            continue
        if pose:
            assert all(r.solved) and min(r.min_eig, default=2.0) > 1.0, ("fixture is not well conditioned", p)
            assert np.abs(T[p, :3, :3] - r.T[:3, :3]).max() < 1e-5, (p, T[p], r.T)
            assert np.abs(T[p, :3, 3] - r.T[:3, 3]).max() < tol_t, (p, T[p], r.T)
        assert np.array_equal(T[p, 3], [0, 0, 0, 1])
        a, b = matched(*data, p)
        assert abs(int(inl[p]) - fo.count_inliers(T[p], a, b, kw.get("inlier_dist", 0.025))) <= 2, p
    return got, want


def planted(counts, outliers, seed, n=None, offset=0.0):
    rng = np.random.default_rng(seed)
    pairs = [po.planted_matches(rng, m, outliers, offset=offset) for m in counts]
    return batch([x[:2] for x in pairs], n=n, seed=seed), [x[2] for x in pairs]


RAGGED = [700, 1000, 333, 1024, 517]


# ---------------------------------------------------------------------------------------------- the tuple list, exactly
@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 12345, 2 ** 63 + 5])
def test_list_and_pose_seed(seed):
    data, _ = planted(RAGGED, 0.3, seed=1, n=1100)
    check(data, seed=seed)


@pytest.mark.gpu
def test_seed_top_bit_reaches_kernel():
    data, _ = planted(RAGGED, 0.3, seed=1, n=1100)
    (_, _, c1, _), _ = check(data, seed=5)
    (_, _, c2, _), _ = check(data, seed=2 ** 63 + 5)
    assert not np.array_equal(c1, c2)


@pytest.mark.gpu
@pytest.mark.parametrize("tuple_scale", [0.9, 0.95, 0.99])
def test_tuple_scale(tuple_scale):
    data, _ = planted(RAGGED, 0.3, seed=2, n=1100)
    check(data, tuple_scale=tuple_scale, seed=3)


@pytest.mark.gpu
@pytest.mark.parametrize("max_tuples", [1, 7, 1000, 1500])
def test_max_tuples(max_tuples):
    # 1: one tuple, too few correspondences for a pose; 1500: a list of 4500 entries, past the shared-memory staging
    data, _ = planted([4000, 3000, 500], 0.3, seed=4, n=4000)
    (_, _, _, ncorr), want = check(data, max_tuples=max_tuples, seed=7, pose=max_tuples >= 1000)
    if max_tuples < 1000:
        assert np.all(ncorr == 3 * max_tuples)
    if max_tuples == 1500:
        assert ncorr[0] == 4500 > STAGE


@pytest.mark.gpu
@pytest.mark.parametrize("m", [3, 9, 10, 4096, 4097, 20011])
@pytest.mark.parametrize("tuple_test", [True, False])
def test_match_counts(m, tuple_test):
    rng = np.random.default_rng(m)
    a, b, _, _ = po.planted_matches(rng, m, 0.3 if m > 10 else 0.0)
    other = po.planted_matches(rng, 800, 0.3)[:2]
    data = batch([other, (a, b)], n=max(m, 800), seed=m)
    # three matches repeated in a list of tuples, or a bare 10: a pose, but not one to compare to 1e-5
    (_, _, _, ncorr), want = check(data, tuple_test=tuple_test, seed=11, pose=m > 10)
    if not tuple_test:
        assert ncorr[1] == m
        assert want[1].posed == (m >= 10)


@pytest.mark.gpu
def test_trials_run_out():
    # 12 and 30 matches give 1200 and 3000 trials, far fewer accepted than max_tuples
    data, _ = planted([12, 30, 600], 0.5, seed=8, n=600)
    (_, _, _, ncorr), want = check(data, seed=2, pose=False)
    assert ncorr[0] < 3000 and ncorr[1] < 3000


# ---------------------------------------------------------------------------------------------- options
@pytest.mark.gpu
@pytest.mark.parametrize("use_absolute_scale", [False, True])
@pytest.mark.parametrize("decrease_mu", [False, True])
@pytest.mark.parametrize("iterations", [0, 1, 64])
def test_options(use_absolute_scale, decrease_mu, iterations):
    data, _ = planted(RAGGED, 0.3, seed=9, n=1100)
    check(data, use_absolute_scale=use_absolute_scale, decrease_mu=decrease_mu, iterations=iterations, seed=1)


@pytest.mark.gpu
@pytest.mark.parametrize("division_factor,max_corr_dist", [(1.4, 0.025), (2.0, 0.05), (1.1, 0.01)])
def test_schedule(division_factor, max_corr_dist):
    data, _ = planted(RAGGED, 0.3, seed=10, n=1100)
    check(data, division_factor=division_factor, max_corr_dist=max_corr_dist, seed=1)


@pytest.mark.gpu
def test_far_from_origin():
    # scan coordinates in metres, 100 units out: the translation is compared to 1e-5 times the coordinate magnitude
    data, _ = planted([800, 1000, 611], 0.3, seed=60, n=1000)
    for x in data[:2]:
        x += np.float32(100.0)
    check(data, tol_t=1e-5 * 101, seed=6)


# ---------------------------------------------------------------------------------------------- ground truth
@pytest.mark.gpu
@pytest.mark.parametrize("outliers", [0.3, 0.5])
def test_recovers_planted_pose(outliers):
    data, gts = planted([300, 1000, 700, 1024], outliers, seed=int(outliers * 100), n=1100)
    (T, inl, _, _), _ = check(data, seed=4)
    for p, gt in enumerate(gts):
        R = T[p, :3, :3].astype(np.float64) @ gt[:3, :3].T
        assert np.degrees(np.arccos(np.clip((np.trace(R) - 1) / 2, -1, 1))) < 0.25, p
        assert np.linalg.norm(T[p, :3, 3] - gt[:3, 3]) < 0.005, p
        assert inl[p] >= (1 - outliers) * data[4][p] * 0.8


# ---------------------------------------------------------------------------------------------- degenerate, ragged
@pytest.mark.gpu
def test_degenerate_pairs_in_one_batch():
    rng = np.random.default_rng(40)
    good = [po.planted_matches(rng, 500, 0.3)[:2] for _ in range(2)]
    few = po.planted_matches(rng, 40, 1.0)[:2]                        # all outliers: few tuples pass
    line = np.zeros((60, 3), np.float32); line[:, 0] = np.arange(60) * 0.125
    pairs = [good[0], (line[:0], line[:0]), (line[:2], line[:2]), few, good[1], (line[:9], line[:9] + 0.5)]
    data = batch(pairs, n=600, seed=41)
    for tuple_test in (True, False):
        (T, inl, _, ncorr), want = check(data, tuple_test=tuple_test, seed=3, pose=False)
        eye = np.eye(4, dtype=np.float32)
        # no pose: 0 and 2 matches; with the tuple test, outliers that give fewer than 10 correspondences; without it,
        # 9 matches (with it, 9 collinear matches pass as many tuples)
        for p in (1, 2, 3 if tuple_test else 5):
            assert np.array_equal(T[p], eye) and inl[p] == 0, p
        assert ncorr[1] == 0 and ncorr[2] == (0 if tuple_test else 2)
        assert ncorr[3] < 10 if tuple_test else ncorr[5] == 9
        assert want[0].posed and want[4].posed


@pytest.mark.gpu
def test_deterministic_and_pairs_independent():
    rng = np.random.default_rng(70)
    pairs = [po.planted_matches(rng, m, 0.4)[:2] for m in (900, 5000, 77)]
    data = batch(pairs, n=5000, seed=71)
    r1 = fgr_call(*data, seed=3)
    r2 = fgr_call(*data, seed=3)
    assert all(np.array_equal(x, y) for x, y in zip(r1, r2))
    for p in range(3):
        other = [x.copy() for x in data]
        src, tgt, idx1, idx2, count = other
        q = [i for i in range(3) if i != p]
        src[q] = rng.uniform(-1, 1, src[q].shape); tgt[q] = rng.uniform(-1, 1, tgt[q].shape)
        idx1[q] = rng.integers(0, 5000, idx1[q].shape); count[q] = rng.integers(0, 5000, len(q))
        r3 = fgr_call(*other, seed=3)
        assert all(np.array_equal(x[p], y[p]) for x, y in zip(r3, r1)), p
    alone = fgr_call(*(x[:1] for x in data), seed=3)                  # pair 0 alone: same bits
    assert all(np.array_equal(x[0], y[0]) for x, y in zip(alone, r1))


# ---------------------------------------------------------------------------------------------- public interface
@pytest.mark.gpu
def test_estimate_poses_mapping():
    import torch
    import ri_b200
    data, _ = planted(RAGGED, 0.3, seed=12, n=1100)
    d = [torch.from_numpy(x).cuda() for x in data]
    T, inl = ri_b200.registration.estimate_poses(*d, func='fgr', voxel_size=0.08, seed=5)
    r = ri_b200.registration.fgr(*d, maximum_correspondence_distance=0.04, inlier_dist=0.08, seed=5,
                                 return_correspondences=True)
    assert torch.equal(T, r['transformation']) and torch.equal(inl, r['inliers'])
    want = replays(*data, max_corr_dist=0.04, inlier_dist=0.08, seed=5)
    corr = r['correspondences'].cpu().numpy()
    for p, w in enumerate(want):
        assert int(r['num_correspondences'][p]) == len(w.corr) and np.array_equal(corr[p, :len(w.corr)], w.corr)
    off = ri_b200.registration.fgr(*d, tuple_test=False, return_correspondences=True)
    c = off['correspondences'].cpu().numpy()
    for p in range(len(RAGGED)):
        assert np.array_equal(c[p, :RAGGED[p]], np.arange(RAGGED[p])) and np.all(c[p, RAGGED[p]:] == -1)
    with pytest.raises(ValueError):
        ri_b200.registration.estimate_poses(*d, func='teaserpp')


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
    meter = ri_b200.registration.MeterModelNet40_registration('fgr', icp=icp)
    meter.update((desc, desc2), (src, tgt, gt))
    r = meter.compute()
    assert set(r) == {'succ', 'rre', 'rte', 'rmse', 'reg_time', 'rmse_succ'}
    assert r['rmse_succ'] == 1.0 and r['rre'] < 0.05 and r['rte'] < 1e-3 and r['rmse'] < 1e-3, r


# ---------------------------------------------------------------------------------------------- argument errors
@pytest.mark.gpu
def test_argument_errors():
    import torch
    import ri_b200  # noqa: F401
    P, n = 3, 40
    f = lambda *s: torch.rand(*s, device="cuda")
    i = lambda *s: torch.zeros(*s, dtype=torch.int32, device="cuda")
    ok = dict(src=f(P, n, 3), tgt=f(P, n + 5, 3), idx1=i(P, n), idx2=i(P, n), count=i(P))
    opts = dict(max_corr_dist=0.025, iterations=64, division_factor=1.4, use_absolute_scale=False, decrease_mu=True,
                tuple_test=True, tuple_scale=0.95, max_tuples=1000, seed=0, inlier_dist=0.025)
    op = torch.ops.ri.fgr
    call = lambda kw, **o: op(kw["src"], kw["tgt"], kw["idx1"], kw["idx2"], kw["count"], *{**opts, **o}.values())
    call(ok)
    bad = [dict(src=f(P, n)), dict(src=f(P, n, 4)), dict(tgt=f(P, n, 2)), dict(tgt=f(P + 1, n, 3)),
           dict(idx1=i(P, n + 1)), dict(idx2=i(P, n - 1)), dict(idx1=i(P - 1, n), idx2=i(P - 1, n)), dict(idx1=i(P, n, 1)),
           dict(count=i(P, 1)), dict(count=i(P + 1)), dict(src=f(P, n, 3).cpu())]
    for b in bad:
        with pytest.raises(RuntimeError):
            call({**ok, **b})
    for o in (dict(max_corr_dist=0.0), dict(max_corr_dist=-1.0), dict(iterations=-1), dict(division_factor=1.0),
              dict(division_factor=0.5), dict(tuple_scale=0.0), dict(tuple_scale=1.01), dict(max_tuples=0),
              dict(max_tuples=2 ** 30), dict(inlier_dist=0.0), dict(inlier_dist=-0.1)):
        with pytest.raises(RuntimeError):
            call(ok, **o)
    big = dict(ok, idx1=i(1, 43 * 10 ** 6), idx2=i(1, 43 * 10 ** 6), src=f(1, n, 3), tgt=f(1, n, 3), count=i(1))
    with pytest.raises(RuntimeError, match="unsupported"):                # 100 * ld >= 2^32: the trial index is 32-bit
        call(big)
    torch.cuda.synchronize()
