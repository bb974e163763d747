"""fp64 replay of csrc/pose.cu (row f3) for the tests only: the same samples, checks, winner rule and refit, one pair at a time.

RANSAC in the kernel, per pair p and hypothesis h < hyps:
    (i0, i1, i2) = sample3(seed, p, h, M)           splitmix64, bit for bit (uint64 with wrap-around)
    hypothesis: edge-length similarity, triangle frames with their 1e-6 norm guards, R = F_b F_a^T, centroid translation,
                every sample point within `thresh` of its partner
    count = #{m : |R a_m + t - b_m| < thresh} over all M matches
    winner = largest count, lowest id on ties; refit = `refine_iters` rounds of {inliers under T -> Kabsch}, stopping (and
    keeping T) when fewer than 3 inliers remain; inliers = the count under the returned T, 0 when no pose was found.
hyps == 0 is one Kabsch over all matches.

The kernel computes the checks in fp32; the replay computes them in fp64 and flags every comparison whose fp64 value lies
within a band of its threshold that fp32 rounding and FMA contraction on the GPU could cross.  A count becomes an interval
[lo, hi] (flagged residuals count toward hi only) and a result is *unambiguous* when it is the same under every resolution
of the flags; the GPU tests check the kernel only on fixtures the replay calls unambiguous.  The band of a comparison is
`rel` relative to its threshold plus an absolute term of `c` fp32 epsilons of the coordinate magnitude, widened for a
hypothesis by the conditioning of its triangle frames.  The product package never imports this module.
"""
from dataclasses import dataclass

import numpy as np

from oracle.cpu_oracle import kabsch

EPS32 = float(np.finfo(np.float32).eps)
MASK64 = (1 << 64) - 1
GUARD = 1e-6                 # tri_frame's norm guard


def mix64(x):
    """splitmix64 finaliser on a Python int or a numpy uint64 array, with explicit 64-bit wrap-around."""
    if isinstance(x, np.ndarray):
        x = x.astype(np.uint64)
        with np.errstate(over="ignore"):
            x = x + np.uint64(0x9E3779B97F4A7C15)
            x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))
    x = (int(x) + 0x9E3779B97F4A7C15) & MASK64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & MASK64
    return x ^ (x >> 31)


def sample3(seed, pair, hyp, M):
    """Three distinct indices in [0, M), M >= 3: the kernel's sample3 on one hypothesis or on an int array of them
    ([H] -> [H, 3] int64)."""
    many = np.ndim(hyp) > 0
    h = np.atleast_1d(np.asarray(hyp, np.int64))
    key = (int(seed) & MASK64) ^ ((int(pair) & MASK64) << 32 & MASK64)
    r0 = mix64(np.uint64(key) ^ (h.astype(np.uint32).astype(np.uint64)))
    r1 = mix64(r0)
    r2 = mix64(r1)
    i0 = (r0 % np.uint64(M)).astype(np.int64)
    i1 = (r1 % np.uint64(M - 1)).astype(np.int64)
    i1 += i1 >= i0
    i2 = (r2 % np.uint64(M - 2)).astype(np.int64)
    lo, hi = np.minimum(i0, i1), np.maximum(i0, i1)
    i2 += i2 >= lo
    i2 += i2 >= hi
    out = np.stack([i0, i1, i2], -1)
    return out if many else tuple(int(v) for v in out[0])


def _near(x, thr, band):
    return np.abs(x - thr) <= band


def _frames(p0, p1, p2, rel, c):
    """tri_frame on [H,3] triangles -> (frame [H,3,3] with e1 e2 e3 as columns, checks [(pass, near)], conditioning [H])."""
    u, v = p1 - p0, p2 - p0
    nu = np.linalg.norm(u, axis=1)
    nv = np.linalg.norm(v, axis=1)
    e1 = u / np.where(nu > 0, nu, 1)[:, None]
    w = v - e1 * np.sum(v * e1, 1)[:, None]
    nw = np.linalg.norm(w, axis=1)
    e2 = w / np.where(nw > 0, nw, 1)[:, None]
    e3 = np.cross(e1, e2)
    # the difference of two fp32 coordinates is correctly rounded, so nu carries a relative error only (coincident points
    # give exactly 0); nw = |v - e1 (v.e1)| cancels and carries an error of the order of |v|
    checks = [(nu > GUARD, _near(nu, GUARD, rel * GUARD + c * EPS32 * nu)),
              (nw > GUARD, _near(nw, GUARD, rel * GUARD + c * EPS32 * nv))]
    cond = 1 + (nu + nv) / np.maximum(np.minimum(nu, nw), GUARD)
    return np.stack([e1, e2, e3], -1), checks, cond


@dataclass
class Hypotheses:
    idx: np.ndarray          # [H,3] sampled match indices
    valid: np.ndarray        # [H] passes every check in fp64
    amb: np.ndarray          # [H] no check fails outside its band and some check lies inside it: the GPU may go either way
    T: np.ndarray            # [H,4,4] fp64 pose of the sample (identity where a frame is degenerate)
    err: np.ndarray          # [H] bound on |fp32 residual - fp64 residual| under this pose


def hypotheses(a, b, hyps, seed, pair, thresh, edge_sim, rel=1e-4, c=16.0):
    """The kernel's hypothesis for h = 0..hyps-1 of pair `pair` on matched coordinates a, b [M,3] (M >= 3)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    idx = sample3(seed, pair, np.arange(hyps), len(a))
    A, B = a[idx], b[idx]                                            # [H, sample point, coordinate]
    e0 = c * EPS32 * _scale(a, b)                                    # rounding of a coordinate difference
    checks = []
    for i, j in ((0, 1), (1, 2), (2, 0)):                            # edge-length similarity, both directions
        ea = np.linalg.norm(A[:, i] - A[:, j], axis=1)
        eb = np.linalg.norm(B[:, i] - B[:, j], axis=1)
        for x, y in ((ea, eb), (eb, ea)):
            checks.append((x >= y * edge_sim, _near(x, y * edge_sim, rel * np.maximum(x, y) + e0)))
    Fa, ca_checks, ca = _frames(A[:, 0], A[:, 1], A[:, 2], rel, c)
    Fb, cb_checks, cb = _frames(B[:, 0], B[:, 1], B[:, 2], rel, c)
    checks += ca_checks + cb_checks
    R = Fb @ np.swapaxes(Fa, 1, 2)
    t = B.mean(1) - np.einsum("hij,hj->hi", R, A.mean(1))
    T = np.tile(np.eye(4), (hyps, 1, 1)); T[:, :3, :3] = R; T[:, :3, 3] = t
    err = e0 * np.maximum(ca, cb)
    d = np.linalg.norm(np.einsum("hij,hkj->hki", R, A) + t[:, None] - B, axis=2)     # [H,3]: the sample's residuals
    checks += [(d[:, k] < thresh, _near(d[:, k], thresh, rel * thresh + err)) for k in range(3)]
    valid = np.all([ok for ok, _ in checks], 0)
    fails = np.any([~ok & ~near for ok, near in checks], 0)
    amb = ~fails & np.any([near for _, near in checks], 0)
    return Hypotheses(idx, valid, amb, T, err)


def _scale(a, b):
    return max(1.0, float(np.abs(a).max(initial=0)), float(np.abs(b).max(initial=0)))


def count_interval(T, a, b, thresh, err, rel=1e-4):
    """Inliers of pose T: (lo, hi) — residuals inside the band count toward hi only."""
    d = np.linalg.norm(np.asarray(a, np.float64) @ np.asarray(T, np.float64)[:3, :3].T + T[:3, 3] - b, axis=1)
    sure = (d < thresh) & ~_near(d, thresh, rel * thresh + err)
    maybe = _near(d, thresh, rel * thresh + err)
    return int(sure.sum()), int(sure.sum() + maybe.sum())


def hypothesis_counts(hy, a, b, thresh, rel=1e-4, chunk=64):
    """[H] lo, hi and the fp64 count of every valid-or-ambiguous hypothesis (0 for certainly invalid ones)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    H = len(hy.valid)
    lo = np.zeros(H, np.int64); hi = np.zeros(H, np.int64); nom = np.zeros(H, np.int64)
    todo = np.nonzero(hy.valid | hy.amb)[0]
    for s in range(0, len(todo), chunk):
        h = todo[s:s + chunk]
        R, t = hy.T[h, :3, :3], hy.T[h, :3, 3]
        d = np.linalg.norm(np.einsum("hij,mj->hmi", R, a) + t[:, None] - b[None], axis=2)     # [h,M]
        band = _near(d, thresh, rel * thresh + hy.err[h, None])
        lo[h] = np.sum((d < thresh) & ~band, 1)
        hi[h] = lo[h] + np.sum(band, 1)
        nom[h] = np.sum(d < thresh, 1)
    lo[hy.amb] = 0                                                    # may be rejected by a check on the GPU
    return lo, hi, nom


@dataclass
class Replay:
    winner: int              # winning hypothesis id, -1 when no hypothesis is valid (and in Kabsch mode)
    winner_lo: int
    winner_hi: int
    unambiguous: bool        # the winner, every refit round's inlier set and the outcome are the same under every flag
    T: np.ndarray            # [4,4] fp64 pose after the refit (identity when no pose was found)
    inliers: int             # nominal count under T
    best_key: int            # what the kernel leaves in best[p]: (inliers << 32) | (0xffffffff - winner), 0 for none


def replay(a, b, hyps, thresh, edge_sim=0.9, refine_iters=3, seed=0, pair=0, rel=1e-4, c=16.0):
    """The kernel's result for one pair: a, b [M,3] are the matched coordinates (src[idx1[:M]], tgt[idx2[:M]])."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    err = c * EPS32 * _scale(a, b)
    if len(a) < 3:
        return Replay(-1, 0, 0, True, np.eye(4), 0, 0)
    if hyps == 0:
        T = kabsch(a, b)
        return Replay(-1, 0, 0, True, T, count_interval(T, a, b, thresh, 0.0, 0.0)[0], 0)
    hy = hypotheses(a, b, hyps, seed, pair, thresh, edge_sim, rel, c)
    lo, hi, nom = hypothesis_counts(hy, a, b, thresh, rel)
    nom = np.where(hy.valid, nom, -1)                                 # the fp64 decisions
    if nom.max() < 0:
        return Replay(-1, 0, 0, not hy.amb.any(), np.eye(4), 0, 0)
    w = int(np.argmax(nom))                                           # the first maximum: lowest id wins ties
    ids = np.arange(hyps)
    rivals = (hy.valid | hy.amb) & (ids != w)
    # a rival with a lower id wins a tie, one with a higher id must exceed the winner's count
    unamb = bool(not hy.amb[w] and np.all(np.where(ids[rivals] < w, hi[rivals] < lo[w], hi[rivals] <= lo[w])))
    # refit from the winning hypothesis; the kernel keeps T in fp32 between rounds
    T = Tf = hy.T[w]
    band = hy.err[w]
    for _ in range(refine_iters):
        d = np.linalg.norm(a @ Tf[:3, :3].T + Tf[:3, 3] - b, axis=1)
        unamb &= not np.any(_near(d, thresh, rel * thresh + band))
        m = d < thresh
        if m.sum() < 3:
            break
        T = kabsch(a[m], b[m])
        Tf = T.astype(np.float32).astype(np.float64)
        band = err
    n = count_interval(Tf, a, b, thresh, 0.0, 0.0)[0]
    return Replay(w, int(lo[w]), int(hi[w]), bool(unamb), T, n, (int(nom[w]) << 32) | (0xFFFFFFFF - w))


# ---------------------------------------------------------------------------------------------- fixtures of the tests
def rand_pose(rng, max_t=0.8):
    ax = rng.standard_normal(3); ax /= np.linalg.norm(ax)
    ang = rng.uniform(0, np.pi)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    T = np.eye(4); T[:3, :3] = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K
    T[:3, 3] = rng.uniform(-max_t, max_t, 3)
    return T


def planted_matches(rng, m, outlier_frac, noise=0.005, offset=0.0, gt=None):
    """m matches of a uniform cloud in [-1, 1]^3 (+ offset) under pose gt, a fraction of them replaced by random partners:
    -> (a [m,3] f32, b [m,3] f32, gt [4,4], outlier mask [m])."""
    gt = rand_pose(rng) if gt is None else gt
    a = rng.uniform(-1, 1, (m, 3)) + offset
    b = a @ gt[:3, :3].T + gt[:3, 3] + rng.normal(0, noise, (m, 3))
    bad = rng.random(m) < outlier_frac
    b[bad] = rng.uniform(-1, 1, (int(bad.sum()), 3)) + offset
    return a.astype(np.float32), b.astype(np.float32), gt, bad
