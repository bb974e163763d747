"""CPU self-test of the FPFH reference (tests/fpfh_oracle.py, row f8): hand-computed pair features, the histogram sums,
rigid invariance, the duplicate-point and n <= 1 cases, and the fp32 distance emulation."""
import numpy as np

import fpfh_oracle as ref

C = np.sqrt(0.5)


def _pf(p1, n1, p2, n2):
    f, _ = ref.pair_features(np.array(p1, np.float32), np.array(n1, np.float32), np.array(p2, np.float32),
                             np.array(n2, np.float32))
    return f


def test_pair_features_by_hand():
    # parallel normals across the segment: no swap, v = dp x n1 = -y, w = n1 x v = +x
    assert np.array_equal(_pf([0, 0, 0], [0, 0, 1], [1, 0, 0], [0, 0, 1]), [0.0, 0.0, 0.0])
    # no swap (acos|a1| = pi/4 < acos|a2| = pi/2): f2 = a1 = sqrt(1/2), f0 = atan2(-c, c)
    assert np.allclose(_pf([0, 0, 0], [C, 0, C], [1, 0, 0], [0, 0, 1]), [-np.pi / 4, 0.0, C], atol=1e-7)
    # swap (acos|a1| = pi/2 > acos|a2| = pi/4): n1' = n2, dp negated, f2 = -a2
    assert np.allclose(_pf([0, 0, 0], [0, 0, 1], [1, 0, 0], [C, 0, C]), [np.pi / 4, 0.0, -C], atol=1e-7)
    # a tilted second normal gives f1 = v.n2 != 0
    n2 = np.array([0.0, 0.6, 0.8])
    assert np.allclose(_pf([0, 0, 0], [0, 0, 1], [1, 0, 0], n2), [np.arctan2(0.0, 0.8), -0.6, 0.0], atol=1e-7)
    # the two zero returns: coincident points, and v = dp x n1' = 0 after the swap
    assert np.array_equal(_pf([1, 2, 3], [0, 0, 1], [1, 2, 3], [1, 0, 0]), [0.0, 0.0, 0.0])
    assert np.array_equal(_pf([0, 0, 0], [0, 0, 1], [1, 0, 0], [1, 0, 0]), [0.0, 0.0, 0.0])
    b, amb = ref.bins(np.zeros(3))
    assert b.tolist() == [5, 5, 5] and not amb.any()
    b, _ = ref.bins(np.array([np.pi, 1.0, -1.0]))                     # the upper edge clamps to bin 10
    assert b.tolist() == [10, 10, 0]


def _cloud(n, seed):
    rng = np.random.default_rng(seed)
    p = rng.standard_normal((n, 3)); p /= np.linalg.norm(p, axis=1, keepdims=True)
    p *= rng.uniform(0.8, 1.2, (n, 1))
    nrm = rng.standard_normal((n, 3)); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return p.astype(np.float32), nrm.astype(np.float32)


def test_histogram_sums():
    p, nrm = _cloud(600, 1)
    idx, cnt = ref.hybrid_lists(p, 0.4, 40)
    fp, sp, c, _ = ref.compute_fpfh(p, nrm, idx, cnt)
    many = cnt > 1
    assert many.mean() > 0.9
    g = c.reshape(-1, 3, 11).sum(2)
    assert (g[many] == (cnt[many] - 1)[:, None]).all() and (g[~many] == 0).all()
    sg = sp.reshape(-1, 3, 11).sum(2)
    assert np.allclose(sg[many], 100.0, rtol=1e-12) and (sg[~many] == 0).all()
    fg = fp.reshape(-1, 3, 11).sum(2)
    assert np.allclose(fg[many], 100.0 + sg[many], rtol=1e-12)         # every weighted sum is non-zero here
    assert (fp[~many] == 0).all()


def test_rigid_invariance():
    p, nrm = _cloud(500, 2)
    idx, cnt = ref.hybrid_lists(p, 0.4, 50)
    rng = np.random.default_rng(3)
    q, r = np.linalg.qr(rng.standard_normal((3, 3))); q *= np.sign(np.diag(r)); q *= np.linalg.det(q)
    p2 = (p.astype(np.float64) @ q.T + rng.standard_normal(3)).astype(np.float32)
    n2 = (nrm.astype(np.float64) @ q.T).astype(np.float32)
    # the rotated copy is rounded to fp32: compare where no bin is within 1e-5 of its edge
    c1, a1 = ref.spfh_counts(p, nrm, idx, cnt, bin_tol=1e-5, swap_tol=1e-5)
    c2, a2 = ref.spfh_counts(p2, n2, idx, cnt, bin_tol=1e-5, swap_tol=1e-5)
    ok = ~(a1 | a2)
    assert ok.mean() > 0.95
    assert np.array_equal(c1[ok], c2[ok])
    f1 = ref.fpfh_from_spfh(p, ref.spfh_from_counts(c1, cnt), idx, cnt)
    f2 = ref.fpfh_from_spfh(p2, ref.spfh_from_counts(c2, cnt), idx, cnt)
    nb_ok = ok & np.array([ok[idx[i, :cnt[i]]].all() for i in range(len(p))])
    assert nb_ok.mean() > 0.5
    assert np.abs(f1[nb_ok] - f2[nb_ok]).max() < 1e-4 * np.abs(f1).max()


def test_duplicates_and_isolated_points():
    p = np.array([[0, 0, 0], [0.1, 0, 0], [0, 0.1, 0], [0, 0, 0.1], [5, 5, 5], [0, 0, 0]], np.float32)
    nrm = np.tile(np.array([[0, 0, 1]], np.float32), (6, 1))
    idx, cnt = ref.hybrid_lists(p, 0.5, 10)
    assert cnt.tolist() == [5, 5, 5, 5, 1, 5]
    assert idx[5, :2].tolist() == [0, 5] and idx[0, :2].tolist() == [0, 5]     # (0, index) keys: 0 first, then 5
    fp, sp, c, _ = ref.compute_fpfh(p, nrm, idx, cnt)
    # q = 5 meets itself at position 1 and q = 0 meets its duplicate: the (0,0,0) feature lands in bins 5, 16, 27
    for q in (0, 5):
        assert c[q, 5] >= 1 and c[q, 16] >= 1 and c[q, 27] >= 1
        assert c[q].reshape(3, 11).sum(1).tolist() == [4, 4, 4]
    assert np.array_equal(c[0], c[5]) and np.allclose(fp[0], fp[5], rtol=0, atol=1e-12)
    # the zero-distance entry carries no weight: FPFH of q = 5 equals the one computed without its self entry
    wo = idx.copy(); wo[5, 1:cnt[5] - 1] = idx[5, 2:cnt[5]]
    f_wo = ref.fpfh_from_spfh(p, sp, wo, cnt - (np.arange(6) == 5))
    assert np.array_equal(fp[5], f_wo[5])
    assert (fp[4] == 0).all() and (sp[4] == 0).all() and (c[4] == 0).all()   # isolated: n = 1
    one = ref.compute_fpfh(p[:1], nrm[:1], *ref.hybrid_lists(p[:1], 1.0, 5))
    assert (one[0] == 0).all()


def test_fp32_distance_emulation():
    rng = np.random.default_rng(4)
    q = rng.standard_normal((20000, 3)).astype(np.float32)
    p = rng.standard_normal((20000, 3)).astype(np.float32)
    d = ref.fp32_dist(q, p)
    assert d.dtype == np.float32
    exact = np.sum((q.astype(np.float64) - p.astype(np.float64)) ** 2, 1)
    assert np.abs(d - exact).max() <= 4e-7 * exact.max()
    # against fp32 rounding of an exactly computed fma chain (Python fractions) on a few hundred inputs
    from fractions import Fraction
    for i in range(300):
        dx, dy, dz = (np.float32(q[i, a] - p[i, a]) for a in range(3))
        a = np.float32(dx * dx)
        b = np.float32(float(Fraction(float(dy)) ** 2 + Fraction(float(a))))
        c = float(Fraction(float(dz)) ** 2 + Fraction(float(b)))
        assert np.float32(c) == d[i] or abs(np.float64(np.float32(c)) - c) == abs(np.float64(d[i]) - c), i
