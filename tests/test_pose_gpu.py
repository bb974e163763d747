"""Row f3 on the GPU: csrc/pose.cu against its fp64 replay (tests/pose_oracle.py).

RANSAC is checked hypothesis by hypothesis: `best[p]` holds (inliers << 32) | (0xffffffff - id) of the winner after the
call (include/ri_b200.h), so the winning id must be the replay's, its count must lie in the replay's [lo, hi], the refit
must be the replay's fp64 refit to 1e-5 and the reported inliers must be the count under the returned pose.  Each fixture
is asserted unambiguous on the CPU first, so a change of data cannot quietly weaken a case.  Then: every match is used
(counts around and far beyond the 4096 matches staged in shared memory at a time), ragged and degenerate pairs, Kabsch on
rank-deficient data, coordinates far from the origin, determinism, pair independence, metric edges and argument errors.
"""
import numpy as np
import pytest

import pose_oracle as ref
from oracle.cpu_oracle import kabsch, registration_metrics as metrics_ref

THRESH = 0.08
CAP = 4096                     # matches staged in shared memory at a time


def _pkg():
    import ri_b200
    return ri_b200


def batch(pairs, n=None, seed=0):
    """[(a [m,3], b [m,3])] -> src [P,n,3], tgt [P,n,3], idx1, idx2 [P,n], count [P]: pair p's match k is
    (src[idx1[k]], tgt[idx2[k]]) = (a[k], b[k]), stored at shuffled rows so that the kernel's gather is exercised."""
    rng = np.random.default_rng(seed)
    n = max(max(len(a) for a, _ in pairs), 3) if n is None else n
    P = len(pairs)
    src = rng.uniform(-1, 1, (P, n, 3)).astype(np.float32); tgt = rng.uniform(-1, 1, (P, n, 3)).astype(np.float32)
    idx1 = np.full((P, n), -1, np.int32); idx2 = np.full((P, n), -1, np.int32); count = np.zeros(P, np.int32)
    for p, (a, b) in enumerate(pairs):
        m = len(a)
        r1, r2 = rng.permutation(n)[:m], rng.permutation(n)[:m]
        src[p, r1], tgt[p, r2] = a, b
        idx1[p, :m], idx2[p, :m], count[p] = r1, r2, m
    return src, tgt, idx1, idx2, count


def pose_call(src, tgt, idx1, idx2, count, hyps, thresh=THRESH, edge_sim=0.9, iters=3, seed=0):
    """The C ABI with our own `best` buffer -> (T [P,4,4] f32, inliers [P] i32, best [P] as Python ints)."""
    import torch
    pkg = _pkg()
    d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (src, tgt, idx1, idx2, count)]
    P, n1, n2, ld = src.shape[0], src.shape[1], tgt.shape[1], idx1.shape[1]
    T = torch.empty((P, 4, 4), dtype=torch.float32, device="cuda")
    inl = torch.empty((P,), dtype=torch.int32, device="cuda")
    best = torch.full((max(P, 1),), -1, dtype=torch.int64, device="cuda")
    rc = pkg._lib.lib.ri_pose_from_matches_f32(*(x.data_ptr() for x in d), P, n1, n2, ld, hyps, thresh, edge_sim, iters,
                                               seed & 0xFFFFFFFFFFFFFFFF, T.data_ptr(), inl.data_ptr(), best.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    return T.cpu().numpy(), inl.cpu().numpy(), [int(v) & 0xFFFFFFFFFFFFFFFF for v in best.cpu().numpy()[:P]]


def matched(src, tgt, idx1, idx2, count, p):
    m = int(count[p])
    return src[p][idx1[p, :m]].astype(np.float64), tgt[p][idx2[p, :m]].astype(np.float64)


def check_against_replay(src, tgt, idx1, idx2, count, hyps, edge_sim=0.9, iters=3, seed=0, tol_t=1e-5):
    want = [ref.replay(*matched(src, tgt, idx1, idx2, count, p), hyps, THRESH, edge_sim, iters, seed, p)
            for p in range(len(count))]
    for p, r in enumerate(want):
        assert r.unambiguous, ("fixture is ambiguous under fp32 rounding: change its data", p)
    T, inl, best = pose_call(src, tgt, idx1, idx2, count, hyps, THRESH, edge_sim, iters, seed)
    for p, r in enumerate(want):
        a, b = matched(src, tgt, idx1, idx2, count, p)
        if hyps > 0:
            if r.winner < 0:
                assert best[p] == 0, p
            else:
                assert 0xFFFFFFFF - (best[p] & 0xFFFFFFFF) == r.winner, (p, best[p] & 0xFFFFFFFF, r.winner)
                assert r.winner < hyps
                assert r.winner_lo <= best[p] >> 32 <= r.winner_hi, (p, best[p] >> 32, r.winner_lo, r.winner_hi)
        assert np.abs(T[p, :3, :3] - r.T[:3, :3]).max() < 1e-5, (p, T[p], r.T)
        assert np.abs(T[p, :3, 3] - r.T[:3, 3]).max() < tol_t, (p, T[p], r.T)
        assert np.array_equal(T[p, 3], [0, 0, 0, 1])
        if r.winner < 0 and hyps > 0:
            assert inl[p] == 0
        else:
            lo, hi = ref.count_interval(T[p].astype(np.float64), a, b, THRESH, 16 * ref.EPS32 * ref._scale(a, b))
            assert lo <= inl[p] <= hi, (p, inl[p], lo, hi)
    return T, inl, best, want


def planted_batch(counts, outliers, seed, n=None, offset=0.0):
    rng = np.random.default_rng(seed)
    pairs = [ref.planted_matches(rng, m, outliers, offset=offset)[:2] for m in counts]
    return batch(pairs, n=n, seed=seed)


RAGGED = [700, 1000, 333, 1024, 517]          # odd P, ragged counts


# ---------------------------------------------------------------------------------------------- replay, exact
@pytest.mark.gpu
@pytest.mark.parametrize("hyps", [1, 127, 129, 1000])
def test_replay_hyps(hyps):
    check_against_replay(*planted_batch(RAGGED, 0.3, seed=hyps, n=1100), hyps, seed=1)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 12345, 2 ** 63 + 5])
def test_replay_seed(seed):
    data = planted_batch(RAGGED, 0.3, seed=7, n=1100)
    check_against_replay(*data, 1000, seed=seed)


@pytest.mark.gpu
def test_replay_seed_top_bit_reaches_kernel():
    data = planted_batch(RAGGED, 0.3, seed=7, n=1100)
    _, _, b1, _ = check_against_replay(*data, 1000, seed=5)
    _, _, b2, _ = check_against_replay(*data, 1000, seed=2 ** 63 + 5)
    assert b1 != b2


@pytest.mark.gpu
@pytest.mark.parametrize("edge_sim", [0.5, 0.9, 0.99])
def test_replay_edge_similarity(edge_sim):
    check_against_replay(*planted_batch(RAGGED, 0.3, seed=21, n=1100), 1000, edge_sim=edge_sim, seed=3)


@pytest.mark.gpu
@pytest.mark.parametrize("iters", [1, 3])
@pytest.mark.parametrize("outliers", [0.3, 0.7])
def test_replay_refine_iters_and_outliers(iters, outliers):
    check_against_replay(*planted_batch(RAGGED, outliers, seed=31, n=1100), 1000, iters=iters, seed=4)


# ---------------------------------------------------------------------------------------------- every match is used
def cap_pairs(m, mode, seed):
    """Matches whose tail (index >= 4096) decides the answer: a fit over the first 4096 alone is far off."""
    rng = np.random.default_rng(seed)
    gt = ref.rand_pose(rng)
    if m <= CAP:
        a, b, _, _ = ref.planted_matches(rng, m, 0.3 if mode == "ransac" else 0.0, gt=gt)
        return a, b
    a, b, _, _ = ref.planted_matches(rng, m, 0.0, gt=gt)
    if mode == "kabsch":
        if m - CAP < 16:
            b[CAP:] = a[CAP:] + 3.0                                   # far-off tail matches pull the fit
        else:
            g1 = ref.rand_pose(rng)                                   # the head follows another pose
            b[:CAP] = (a[:CAP] @ g1[:3, :3].T + g1[:3, 3]).astype(np.float32)
    else:
        if m - CAP < 16:
            b[CAP:] = (a[CAP:] @ gt[:3, :3].T + gt[:3, 3]).astype(np.float32)    # exact inliers the count must see
        else:
            b[:CAP] = rng.uniform(-1, 1, (CAP, 3)).astype(np.float32)             # the head is all outliers
    return a, b


@pytest.mark.gpu
@pytest.mark.parametrize("m", [3, 4095, 4096, 4097, 20011])
def test_kabsch_uses_every_match(m):
    a, b = cap_pairs(m, "kabsch", seed=m)
    data = batch([(a, b), cap_pairs(1000, "kabsch", seed=1)], n=max(m, 1000), seed=m)
    T, inl, _ = pose_call(*data, hyps=0)
    want = kabsch(a, b)
    if m > CAP:
        assert np.abs(kabsch(a[:CAP], b[:CAP]) - want).max() > 1e-3       # the tail matters
    assert np.abs(T[0] - want).max() < 1e-5, (T[0], want)
    assert inl[0] == ref.count_interval(T[0].astype(np.float64), a, b, THRESH, 0.0, 0.0)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("m", [3, 4095, 4096, 4097, 20011])
def test_ransac_uses_every_match(m):
    a, b = cap_pairs(m, "ransac", seed=m)
    data = batch([cap_pairs(900, "ransac", seed=2), (a, b)], n=max(m, 900), seed=m)
    T, inl, best, want = check_against_replay(*data, 1000, seed=9)
    assert want[1].winner >= 0
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    lo, hi = ref.count_interval(T[1].astype(np.float64), a64, b64, THRESH, 16 * ref.EPS32)
    assert lo == hi == inl[1]                                          # exact recount over all matches
    if m > CAP + 16:
        assert inl[1] > CAP


# ---------------------------------------------------------------------------------------------- ragged and degenerate
@pytest.mark.gpu
@pytest.mark.parametrize("hyps", [0, 1000])
def test_ragged_and_degenerate_pairs_in_one_batch(hyps):
    rng = np.random.default_rng(40)
    line = np.zeros((60, 3), np.float32); line[:, 0] = np.arange(60) * 0.125
    same = np.full((60, 3), 0.25, np.float32)
    good = [ref.planted_matches(rng, 500, 0.3)[:2] for _ in range(3)]
    n = 600
    pairs = [good[0], (line[:0], line[:0]), good[1], (line[:1], line[:1]), (line[:2], line[:2]), good[2], (line, line + 0.5),
             (same, same + 0.5)]
    src, tgt, idx1, idx2, count = batch(pairs, n=n, seed=41)
    for x in (idx1, idx2):                                             # pair 2: random extra matches up to ld = n,
        x[2, 500:] = np.setdiff1d(np.arange(n), x[2, :500])            # then a count beyond ld, clamped to ld
    count[2] = n + 50
    T, inl, best = pose_call(src, tgt, idx1, idx2, count, hyps)
    eye = np.eye(4, dtype=np.float32)
    for p in (1, 3, 4):
        assert np.array_equal(T[p], eye) and inl[p] == 0, p
    if hyps:
        for p in (6, 7):                                               # collinear, coincident: no valid hypothesis
            assert np.array_equal(T[p], eye) and inl[p] == 0 and best[p] == 0, p
        for p in (1, 3, 4):
            assert best[p] == 0
    ctr = count.copy(); ctr[2] = n
    for p in (0, 2, 5):
        a, b = matched(src, tgt, idx1, idx2, ctr, p)
        r = ref.replay(a, b, hyps, THRESH, 0.9, 3, 0, p)
        assert r.unambiguous
        assert np.abs(T[p] - r.T).max() < 1e-5, p
        lo, hi = ref.count_interval(T[p].astype(np.float64), a, b, THRESH, 16 * ref.EPS32)
        assert lo <= inl[p] <= hi


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["coincident", "collinear", "coplanar"])
def test_kabsch_rank_deficient(kind):
    rng = np.random.default_rng(50)
    m = 80
    if kind == "coincident":
        a = np.tile([0.3, -0.2, 0.1], (m, 1))
    elif kind == "collinear":
        a = np.outer(rng.uniform(-1, 1, m), [0.6, 0.0, 0.8]) + [0.1, 0.2, 0.3]
    else:
        a = rng.uniform(-1, 1, (m, 3)); a[:, 2] = 0.5
    gt = ref.rand_pose(rng)
    a = a.astype(np.float32)
    b = (a @ gt[:3, :3].T + gt[:3, 3]).astype(np.float32)
    T, inl, _ = pose_call(*batch([(a, b)], seed=51), hyps=0)
    R = T[0, :3, :3].astype(np.float64)
    assert np.allclose(R @ R.T, np.eye(3), atol=1e-6) and abs(np.linalg.det(R) - 1) < 1e-6
    res = lambda M: np.linalg.norm(a.astype(np.float64) @ M[:3, :3].T + M[:3, 3] - b)
    want = kabsch(a, b)
    assert res(T[0].astype(np.float64)) <= res(want) * (1 + 1e-5) + 1e-5
    assert inl[0] == m


# ---------------------------------------------------------------------------------------------- far from the origin
@pytest.mark.gpu
@pytest.mark.parametrize("hyps", [0, 1000])
def test_far_from_origin(hyps):
    # scan coordinates in metres, 100 units out: an fp32 coordinate there is only good to ~8e-6, so the translation is
    # compared to 1e-5 times the coordinate magnitude (the rotation keeps 1e-5), and the replay widens its bands likewise
    data = planted_batch([800, 1000, 611], 0.3, seed=60, n=1000, offset=100.0)
    if hyps:
        check_against_replay(*data, hyps, seed=6, tol_t=1e-5 * 101)
    else:
        T, inl, _ = pose_call(*data, hyps=0)
        for p in range(3):
            a, b = matched(*data, p)
            want = kabsch(a, b)
            assert np.abs(T[p, :3, :3] - want[:3, :3]).max() < 1e-5
            assert np.abs(T[p, :3, 3] - want[:3, 3]).max() < 1e-5 * 101


# ---------------------------------------------------------------------------------------------- determinism, independence
@pytest.mark.gpu
@pytest.mark.parametrize("hyps", [0, 1000])
def test_deterministic_and_pairs_independent(hyps):
    rng = np.random.default_rng(70)
    pairs = [ref.planted_matches(rng, m, 0.4)[:2] for m in (900, 5000, 77)]
    data = batch(pairs, n=5000, seed=71)
    r1 = pose_call(*data, hyps, seed=3)
    r2 = pose_call(*data, hyps, seed=3)
    assert all(np.array_equal(x, y) for x, y in zip(r1, r2))
    for p in range(3):
        other = [x.copy() for x in data]
        src, tgt, idx1, idx2, count = other
        q = [i for i in range(3) if i != p]
        src[q] = rng.uniform(-1, 1, src[q].shape); tgt[q] = rng.uniform(-1, 1, tgt[q].shape)
        idx1[q] = rng.integers(0, 5000, idx1[q].shape); count[q] = rng.integers(0, 5000, len(q))
        r3 = pose_call(*other, hyps, seed=3)
        assert np.array_equal(r3[0][p], r1[0][p]) and r3[1][p] == r1[1][p] and r3[2][p] == r1[2][p], p


# ---------------------------------------------------------------------------------------------- registration_metrics
@pytest.mark.gpu
def test_metrics_edges():
    import torch
    pkg = _pkg()
    rng = np.random.default_rng(80)
    gt = np.stack([np.eye(4), np.eye(4), ref.rand_pose(rng)]).astype(np.float32)
    est = gt.copy()
    est[0, :3, :3] = np.diag([-1.0000001, -1.0000001, 1.0])           # 180 degrees with the trace just below -1: clamp
    est[1, :3, :3] = np.diag([-1.0, 1.0, -1.0])                       # 180 degrees exactly
    est[2, :3, 3] += [0.3, 0.0, -0.4]
    cu = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    for n in (0, 17):
        pts = rng.uniform(-1, 1, (3, n, 3)).astype(np.float32)
        got = pkg.registration.registration_metrics(cu(gt), cu(est), cu(pts)).cpu().numpy()
        want = metrics_ref(gt.astype(np.float64), est.astype(np.float64), pts.astype(np.float64)) if n else None
        assert np.all(np.isfinite(got))
        assert abs(got[0, 0] - 180.0) < 1e-9 and abs(got[1, 0] - 180.0) < 1e-9
        # equal fp32 rotations: acos near 1 turns the last bits of the trace into up to ~0.03 degrees
        assert abs(got[2, 1] - 0.5) < 1e-6 and abs(got[2, 0]) < 0.05
        if n == 0:
            assert np.all(got[:, 2] == 0.0)
        else:
            assert np.allclose(got[:, 1:], want[:, 1:], rtol=1e-9, atol=1e-12)
            assert np.allclose(got[:2, 0], want[:2, 0], rtol=1e-12)
    one = pkg.registration.registration_metrics(cu(gt[2:]), cu(est[2:]), cu(pts[2:])).cpu().numpy()
    assert one.shape == (1, 3) and np.array_equal(one[0], got[2])


# ---------------------------------------------------------------------------------------------- argument errors
@pytest.mark.gpu
def test_argument_errors():
    import torch
    P, n = 3, 40
    f = lambda *s: torch.rand(*s, device="cuda")
    i = lambda *s: torch.zeros(*s, dtype=torch.int32, device="cuda")
    ok = dict(src=f(P, n, 3), tgt=f(P, n + 5, 3), idx1=i(P, n), idx2=i(P, n), count=i(P))
    op = torch.ops.ri.pose_from_matches
    call = lambda kw, hyps=100, dist=0.08, iters=3: op(kw["src"], kw["tgt"], kw["idx1"], kw["idx2"], kw["count"], hyps,
                                                       dist, 0.9, iters, 0)
    call(ok)
    bad = [dict(src=f(P, n)), dict(src=f(P, n, 4)), dict(tgt=f(P, n, 2)), dict(tgt=f(P + 1, n, 3)),
           dict(idx1=i(P, n + 1)), dict(idx2=i(P, n - 1)), dict(idx1=i(P - 1, n), idx2=i(P - 1, n)), dict(idx1=i(P, n, 1)),
           dict(count=i(P, 1)), dict(count=i(P + 1)), dict(count=i(1))]
    for b in bad:
        with pytest.raises(RuntimeError):
            call({**ok, **b})
    for kw in (dict(iters=0), dict(iters=-1), dict(dist=0.0), dict(dist=-0.1), dict(hyps=0, iters=0)):
        with pytest.raises(RuntimeError):
            call(ok, **kw)
    torch.cuda.synchronize()
