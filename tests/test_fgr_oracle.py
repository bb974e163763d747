"""CPU self-test of tests/fgr_oracle.py, the fp64 replay that csrc/fgr.cu (row f7) is checked against: its sampler is the
pose sampler's hash chain, its tuple list is the sequential loop's, its GNC solves what it claims to solve, and it recovers
planted poses at the outlier rates the GPU tests use."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import fgr_oracle as fo
import pose_oracle as po
from oracle.cpu_oracle import kabsch


@pytest.mark.parametrize("seed", [0, 77, 2 ** 63 + 5])
def test_trial_stream_is_the_sample3_chain(seed):
    M, pair = 1237, 5
    t = np.arange(4000)
    got = fo.trial_indices(seed, pair, M, t)
    assert np.array_equal(got[:, 0], po.sample3(seed, pair, t, M)[:, 0])     # sample3 takes i0 = r0 % M unchanged
    for h in (0, 1, 999, 3999):
        r0 = po.mix64((seed & po.MASK64) ^ ((pair << 32) & po.MASK64) ^ h)
        r1 = po.mix64(r0)
        r2 = po.mix64(r1)
        assert tuple(got[h]) == (r0 % M, r1 % M, r2 % M)


def _sequential_list(a, b, seed, pair, s, max_tuples):
    """Open3D's loop, trial by trial (scalar Python arithmetic on fp64)."""
    M = len(a)
    a = np.asarray(a, np.float32).astype(np.float64); b = np.asarray(b, np.float32).astype(np.float64)
    s = float(np.float32(s))
    out = []
    for t in range(100 * M):
        idx = fo.trial_indices(seed, pair, M, [t])[0]
        ok = True
        for i, j in ((0, 1), (1, 2), (2, 0)):
            la = np.sqrt(sum((a[idx[i], k] - a[idx[j], k]) ** 2 for k in range(3)))
            lb = np.sqrt(sum((b[idx[i], k] - b[idx[j], k]) ** 2 for k in range(3)))
            ok = ok and la * s < lb and lb < la / s
        if ok:
            out.extend(idx)
            if len(out) == 3 * max_tuples:
                break
    return np.array(out, np.int64)


@pytest.mark.parametrize("max_tuples", [1, 7, 1000])
def test_tuple_list_is_the_sequential_loop(max_tuples):
    rng = np.random.default_rng(3)
    a, b, _, _ = po.planted_matches(rng, 40, 0.5)
    got = fo.tuple_list(a, b, 9, 2, 0.95, max_tuples, chunk=97)      # an odd chunk: the list must not depend on it
    want = _sequential_list(a, b, 9, 2, 0.95, max_tuples)
    assert np.array_equal(got, want)
    assert len(got) % 3 == 0 and 0 < len(got) <= 3 * max_tuples
    idx = got.reshape(-1, 3)
    assert np.all(fo.tuple_accept(a, b, idx, 0.95))
    if max_tuples < 1000:
        assert len(got) == 3 * max_tuples
    else:
        assert len(got) < 3 * max_tuples                              # the 4000 trials run out first
    # trial order: each accepted trial is the next accepted one of the stream
    t = np.arange(100 * len(a))
    acc = fo.trial_indices(9, 2, len(a), t)
    acc = acc[fo.tuple_accept(a, b, acc, 0.95)]
    assert np.array_equal(idx, acc[:len(idx)])


def test_repeated_index_never_passes():
    a = np.random.default_rng(4).uniform(-1, 1, (2, 3)).astype(np.float32)
    assert len(fo.tuple_list(a, a, 0, 0)) == 0
    idx = np.array([[0, 0, 1], [1, 0, 1], [0, 1, 1]])
    assert not fo.tuple_accept(a, a, idx, 0.95).any()


def test_noise_free_recovers_the_planted_pose():
    rng = np.random.default_rng(5)
    a, b, gt, _ = po.planted_matches(rng, 400, 0.0, noise=0.0)
    r = fo.replay(a, b, a, b, seed=1)
    assert r.posed and all(r.solved)
    want = kabsch(a, b)
    assert np.abs(r.T - want).max() < 1e-9, np.abs(r.T - want).max()
    assert np.abs(r.T - gt).max() < 1e-5


def test_gn_step_is_the_linearisation():
    rng = np.random.default_rng(6)
    p = rng.uniform(-1, 1, (50, 3)); qh = rng.uniform(-1, 1, (50, 3))
    Tp = po.rand_pose(rng, 0.3)
    par = 0.3
    JTJ, JTr = fo.normal_equations(p, qh, Tp, par)
    q = qh @ Tp[:3, :3].T + Tp[:3, 3]
    w = (par / (np.sum((p - q) ** 2, 1) + par)) ** 2

    def res(x):                                                       # sqrt(w) (p - Delta(x) q), weights held fixed
        D = fo.delta(x)
        return ((p - (q @ D[:3, :3].T + D[:3, 3])) * np.sqrt(w)[:, None]).reshape(-1)

    h = 1e-6
    Jn = np.stack([(res(h * e) - res(-h * e)) / (2 * h) for e in np.eye(6)], 1)
    assert np.allclose(Jn.T @ Jn, JTJ, rtol=1e-6, atol=1e-6)
    assert np.allclose(Jn.T @ res(np.zeros(6)), JTr, rtol=1e-6, atol=1e-6)
    x = fo.gn_step(JTJ, JTr)
    assert np.allclose(JTJ @ x, -JTr, atol=1e-9)


def test_euler_composition_is_zyx():
    rng = np.random.default_rng(7)
    for x in rng.uniform(-np.pi, np.pi, (20, 3)):
        want = Rotation.from_euler('ZYX', [x[2], x[1], x[0]]).as_matrix()
        assert np.allclose(fo.euler_zyx(*x), want, atol=1e-14)


def test_singular_system_keeps_identity():
    assert fo.gn_step(np.zeros((6, 6)), np.ones(6)) is None
    assert fo.gn_step(np.diag([1, 1, 1, 1, 1, -1.0]), np.ones(6)) is None


def rot_err_deg(T, G):
    c = (np.trace(T[:3, :3] @ G[:3, :3].T) - 1) / 2
    return np.degrees(np.arccos(np.clip(c, -1, 1)))


# thresholds of the GPU tests' planted fixtures: matches of a [-1, 1]^3 cloud, 5 mm noise
RECOVER_DEG, RECOVER_T = 0.25, 0.005


@pytest.mark.parametrize("outliers", [0.3, 0.5])
@pytest.mark.parametrize("m", [300, 1000])
def test_planted_outliers_recover_ground_truth(outliers, m):
    rng = np.random.default_rng(int(outliers * 10) + m)
    for k in range(3):
        a, b, gt, bad = po.planted_matches(rng, m, outliers)
        r = fo.replay(a, b, a, b, seed=k, pair=k)
        assert r.posed and all(r.solved) and min(r.min_eig) > 1.0
        assert rot_err_deg(r.T, gt) < RECOVER_DEG and np.linalg.norm(r.T[:3, 3] - gt[:3, 3]) < RECOVER_T
        assert r.inliers == int((~bad).sum())                        # 5 mm noise, 25 mm radius: every true match


def test_too_few_correspondences_is_no_pose():
    rng = np.random.default_rng(8)
    a, b, _, _ = po.planted_matches(rng, 9, 0.0)
    r = fo.replay(a, b, a, b, tuple_test=False)
    assert not r.posed and np.array_equal(r.T32, np.eye(4, dtype=np.float32)) and r.inliers == 0
    a, b, _, _ = po.planted_matches(rng, 10, 0.0)
    r = fo.replay(a, b, a, b, tuple_test=False)
    assert r.posed and len(r.corr) == 10
