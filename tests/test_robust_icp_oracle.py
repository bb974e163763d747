"""CPU self-test of tests/robust_icp_oracle.py, the fp64 reference that tests/test_robust_icp_gpu.py holds csrc/icp.cu's
robust kernels (row f11) to: the weight table, the L2 limit against the existing oracles, the per-row sum against the
A = W diag(w) W form and W's closed form, and an outlier fixture on which a robust kernel matters."""
import numpy as np
import pytest

import gicp_oracle as go
import icp_oracle
import robust_icp_oracle as ro
from test_gicp_oracle import _pose, _pose_err

# The outlier fixture: on seeds 0 and 2 the oracle's Tukey reaches the ground truth within these bounds and L2 does not
# (L2 ends 0.20 / 0.36 degrees and 16 / 15 mm off; Tukey 0.07 / 0.02 degrees and 1.7 / 1.3 mm for point-to-plane).  On
# seed 1 point-to-plane Tukey diverges (fitness 0.59), so it is not part of the fixture.
OUTLIER_SEEDS = (0, 2)
OUTLIER_R = 0.1
OUTLIER_PLANE_KERNEL = ('tukey', 0.01)                 # 5 sigma of the target's 2 mm noise
OUTLIER_GICP_KERNEL = ('tukey', 0.01 / np.sqrt(2e-3))  # the same along a shared normal, in whitened units (eps = 1e-3)
ROBUST_BOUND = (0.15, 0.005)                           # (degrees, metres) the robust kernel stays within
L2_MISS = 0.01                                         # metres L2's translation error exceeds


def moved_patch_scan(n, seed, frac=0.3, shift=0.05, noise=0.002):
    """A synth.make_scan scene and its copy under a known SE(3) + noise, with the 30 % of the points nearest a random point
    (a piece of furniture) moved by `shift` in a random direction before the motion; init 3 degrees / 3 cm off.
    -> (src, tgt, src_normals, tgt_normals [n,3] fp64, G [4,4], init [4,4])."""
    import ri_b200
    rng = np.random.default_rng(seed)
    S = ri_b200.synth.make_scan(n, seed=seed)
    s = S[:3].T.astype(np.float64); nrm = S[3:].T.astype(np.float64)
    c = s[rng.integers(n)]
    idx = np.argsort(np.linalg.norm(s - c, axis=1))[: int(frac * n)]
    moved = s.copy()
    v = rng.standard_normal(3); moved[idx] += v / np.linalg.norm(v) * shift
    G = _pose(rng, 10.0, 0.2)
    t = moved @ G[:3, :3].T + G[:3, 3] + rng.standard_normal(s.shape) * noise
    init = _pose(rng, 3.0, 0.03) @ G
    return s, t, nrm, nrm @ G[:3, :3].T, G, init


def test_weight_table():
    k = 0.5
    r = np.array([0.0, k / 2, -k / 2, k, -k, 2 * k])
    want = {
        'l2': [1, 1, 1, 1, 1, 1],
        'l1': [0, 4, 4, 2, 2, 1],
        'huber': [1, 1, 1, 1, 1, 0.5],
        'cauchy': [1, 0.8, 0.8, 0.5, 0.5, 0.2],
        'gm': [2, 0.5 / 0.5625 ** 2, 0.5 / 0.5625 ** 2, 0.5 / 0.75 ** 2, 0.5 / 0.75 ** 2, 0.5 / 1.5 ** 2],
        'tukey': [1, 0.5625, 0.5625, 0, 0, 0],
    }
    for name, w in want.items():
        got = ro.weight(name if name in ('l2', 'l1') else (name, k), r)
        assert np.allclose(got, w, rtol=1e-15, atol=0), (name, got)


def test_huber_exactly_one_and_tukey_exactly_zero():
    rng = np.random.default_rng(0)
    k = 0.037
    e = rng.uniform(0, k, 1000) * rng.choice([-1, 1], 1000)
    assert (ro.weight(('huber', k), np.append(e, [k, -k])) == 1.0).all()
    assert (ro.weight(('huber', 1e30), rng.standard_normal(100)) == 1.0).all()
    far = np.append(k + rng.uniform(0, 1, 1000), [k, -k])
    assert (ro.weight(('tukey', k), far * rng.choice([-1, 1], 1002)) == 0.0).all()


def _scan(n, seed, noise=0.002):
    import ri_b200
    rng = np.random.default_rng(seed)
    S = ri_b200.synth.make_scan(n, seed=seed)
    s = S[:3].T.astype(np.float64); nrm = S[3:].T.astype(np.float64)
    G = _pose(rng, 10.0, 0.2)
    t = s @ G[:3, :3].T + G[:3, 3] + rng.standard_normal(s.shape) * noise
    return s, t, nrm, nrm @ G[:3, :3].T, G, _pose(rng, 3.0, 0.03) @ G


def test_l2_equals_existing_oracles():
    s, t, ns, nt, G, init = _scan(3000, seed=5)
    a = ro.icp_point_to_plane(s, t, nt, 0.1, 'l2', init)
    b = icp_oracle.icp_point_to_plane(s, t, nt, 0.1, init)
    assert a[3] == b[3] and np.array_equal(a[4], b[4])
    assert np.abs(a[0] - b[0]).max() < 1e-12 and abs(a[1] - b[1]) < 1e-12 and abs(a[2] - b[2]) < 1e-12
    a = ro.generalized_icp_normals(s, t, ns, nt, 0.1, 'l2', 1e-3, init)
    b = go.generalized_icp_normals(s, t, ns, nt, 0.1, 1e-3, init, form='sqrt')
    assert a[3] == b[3] and np.array_equal(a[4], b[4])
    assert np.abs(a[0] - b[0]).max() < 1e-12 and abs(a[1] - b[1]) < 1e-12 and abs(a[2] - b[2]) < 1e-12


def _closed_form_W(a, b, eps):
    """csrc/icp.cu's closed form of (M^-1)^(1/2), M = 2I - (1 - eps)(a a^T + b b^T), a and b unit or zero."""
    c, r2 = 1.0 - eps, 2.0 ** -0.5
    W = r2 * np.eye(3)
    za, zb = not a.any(), not b.any()
    if not za and not zb:
        s = a @ b
        for sg in (1.0, -1.0):
            u = a + sg * b
            if u @ u > 0:
                W += (1.0 / np.sqrt(2.0 - c * (1.0 + sg * s)) - r2) / (u @ u) * np.outer(u, u)
    elif not (za and zb):
        u = b if za else a
        W += (1.0 / np.sqrt(2.0 - c) - r2) * np.outer(u, u)
    return W


@pytest.mark.parametrize("eps", [1e-3, 0.1, 1.0])
def test_per_row_sum_equals_A_form_and_closed_form(eps):
    rng = np.random.default_rng(1)
    m = 400
    q = rng.uniform(-1, 1, (m, 3)); t = q + rng.normal(0, 0.05, (m, 3))
    unit = lambda x: x / np.linalg.norm(x, axis=1, keepdims=True)
    a = unit(rng.standard_normal((m, 3))); b = unit(rng.standard_normal((m, 3)))
    b[:20] = a[:20]; b[20:40] = -a[20:40]; a[40:60] = 0; b[60:80] = 0; a[80:90] = 0; b[80:90] = 0
    M = 2 * np.eye(3)[None] - (1 - eps) * (a[:, :, None] * a[:, None, :] + b[:, :, None] * b[:, None, :])
    W = ro.whitening(M)
    Wc = np.stack([_closed_form_W(a[i], b[i], eps) for i in range(m)])
    assert np.abs(W - Wc).max() < 1e-12 * np.abs(W).max()
    Ct = np.eye(3)[None] - (1 - eps) * b[:, :, None] * b[:, None, :]
    Cs = M - Ct                                          # = I - (1 - eps) a a^T
    d = q - t
    J0 = go.jacobian0(q)
    for kernel in ('l2', 'l1', ('huber', 0.02), ('cauchy', 0.02), ('gm', 4e-4), ('tukey', 0.05)):
        H, g = ro.gicp_moments(q, t, Cs, Ct, kernel)
        w = ro.weight(kernel, np.einsum('mij,mj->mi', Wc, d))
        A = Wc @ (w[:, :, None] * Wc)
        HA = np.einsum('mka,mkl,mlb->ab', J0, A, J0)
        gA = np.einsum('mka,mkl,ml->a', J0, A, d)
        assert np.abs(H - HA).max() <= 1e-12 * max(1.0, np.abs(HA).max()), kernel
        assert np.abs(g - gA).max() <= 1e-12 * max(1.0, np.abs(gA).max()), kernel
    Hl, gl = go.moments(q, t, Cs, Ct, form='inv')
    H2, g2 = ro.gicp_moments(q, t, Cs, Ct, 'l2')
    assert np.abs(H2 - Hl).max() <= 1e-10 * np.abs(Hl).max() and np.abs(g2 - gl).max() <= 1e-10 * np.abs(Hl).max()


@pytest.mark.parametrize("seed", OUTLIER_SEEDS)
def test_outlier_fixture_needs_a_robust_kernel(seed):
    s, t, ns, nt, G, init = moved_patch_scan(5000, seed)
    l2 = ro.icp_point_to_plane(s, t, nt, OUTLIER_R, 'l2', init)
    tk = ro.icp_point_to_plane(s, t, nt, OUTLIER_R, OUTLIER_PLANE_KERNEL, init)
    assert _pose_err(l2[0], G)[1] > L2_MISS
    rre, rte = _pose_err(tk[0], G)
    assert rre < ROBUST_BOUND[0] and rte < ROBUST_BOUND[1], (rre, rte)
    l2 = ro.generalized_icp_normals(s, t, ns, nt, OUTLIER_R, 'l2', 1e-3, init)
    tk = ro.generalized_icp_normals(s, t, ns, nt, OUTLIER_R, OUTLIER_GICP_KERNEL, 1e-3, init)
    assert _pose_err(l2[0], G)[1] > L2_MISS
    rre, rte = _pose_err(tk[0], G)
    assert rre < ROBUST_BOUND[0] and rte < ROBUST_BOUND[1], (rre, rte)
