"""numpy fp64 replay of the ISS keypoint contract (include/ri_b200.h, ri_iss_keypoints_f32), radius searches by
scipy.spatial.cKDTree.

The kernel's distance is one fp32 expression, fma(dz,dz, fma(dy,dy, dx*dx)); numpy emulates each fma with an exact fp64
product and a double rounding, so the radius cut can differ in the last bit.  Every decision that sits near a boundary is
flagged instead of trusted: per point, `amb` is True when any of these holds for q or for a point q's keypoint test reads
  - a neighbour distance within 1e-6 relative of r^2 (either radius);
  - a ratio e2/e1, e3/e2 within 1e-9 of its gamma, or e3 within 1e-9 e1 of 0 (the sign of s);
  - max |C_ij| within 1e-6 relative of the 1e-12 zero threshold;
  - a suppression comparison with |s(p) - s(q)| <= 1e-9 max(e1(p), e1(q)) between points at different coordinates
    (duplicates have identical neighbourhoods and identical sums, in the kernel and here).
Outside flagged points the kernel's keypoint lists must equal the oracle's exactly.
"""
import numpy as np
from scipy.spatial import cKDTree

RATIO_TOL = 1e-9
DIST_TOL = 1e-6


def fp32_dist(q, p):
    """The kernel's d(q, p) for rows q [m,3], p [m,3] float32 -> float32 [m]."""
    dx, dy, dz = (q.astype(np.float32) - p.astype(np.float32)).T
    a = dx * dx                                                     # fp32, correctly rounded
    b = (dy.astype(np.float64) * dy + a).astype(np.float32)         # fma: exact product, then (double) rounding
    return (dz.astype(np.float64) * dz + b).astype(np.float32)


def resolution(X):
    """X [N,3] float32 -> (res fp64, number of points counted): the mean over finite points of sqrt(d) to the nearest
    other point (duplicates give 0)."""
    F = np.flatnonzero(np.isfinite(X).all(1))
    if len(F) < 2:
        return 0.0, 0
    k = min(8, len(F))
    _, cand = cKDTree(X[F].astype(np.float64)).query(X[F].astype(np.float64), k=k)
    qi = np.repeat(F, k)
    pj = F[cand.reshape(-1)]
    d = fp32_dist(X[qi], X[pj]).astype(np.float64)
    d[qi == pj] = np.inf
    dmin = d.reshape(len(F), k).min(1)
    return float(np.sqrt(dmin).sum() / len(F)), len(F)


def auto_radii(X):
    res, _ = resolution(X)
    return np.float32(6.0 * res), np.float32(4.0 * res)


def radius_pairs(X, F, tree, r):
    """(qi, pj) of every pair with d(q, p) < r*r (fp32), q ascending and p ascending per q; and per point the flag
    'a neighbour distance lies within DIST_TOL of r^2'."""
    N = len(X)
    r2 = np.float32(r) * np.float32(r)
    near = np.zeros(N, bool)
    if r2 <= 0 or len(F) == 0:
        e = np.zeros(0, np.int64)
        return e, e, near
    lists = tree.query_ball_point(X[F].astype(np.float64), float(r) * (1 + 1e-5) + 1e-30, return_sorted=True)
    lens = np.fromiter((len(l) for l in lists), np.int64, len(lists))
    qi = np.repeat(F, lens)
    pj = F[np.concatenate([np.asarray(l, np.int64) for l in lists])] if lens.sum() else np.zeros(0, np.int64)
    d = fp32_dist(X[qi], X[pj])
    close = np.abs(d.astype(np.float64) - np.float64(r2)) <= DIST_TOL * np.float64(r2)
    near[qi[close]] = True
    keep = d < r2
    return qi[keep], pj[keep], near


def iss(X, salient_radius=0.0, non_max_radius=0.0, gamma_21=0.975, gamma_32=0.975, min_neighbors=5):
    """X [N,3] float32 -> dict(idx (ascending keypoints), saliency [N], e1 [N], amb [N] bool, radii (r_s, r_nm) float32)."""
    X = np.ascontiguousarray(X, np.float32)
    N = len(X)
    if salient_radius == 0 or non_max_radius == 0:
        rs, rnm = auto_radii(X)
    else:
        rs, rnm = np.float32(salient_radius), np.float32(non_max_radius)
    finite = np.isfinite(X).all(1)
    F = np.flatnonzero(finite)
    tree = cKDTree(X[F].astype(np.float64)) if len(F) else None
    X64 = X.astype(np.float64)

    # saliency
    qi, pj, near_s = radius_pairs(X, F, tree, rs)
    cnt = np.bincount(qi, minlength=N)
    E = X64[pj] - X64[qi]
    starts = np.concatenate([[0], np.cumsum(cnt)[:-1]])
    has = cnt > 0
    S1 = np.zeros((N, 3)); S2 = np.zeros((N, 3, 3))
    if len(qi):
        S1[has] = np.add.reduceat(E, starts[has], axis=0)
        S2[has] = np.add.reduceat(E[:, :, None] * E[:, None, :], starts[has], axis=0)
    n = np.maximum(cnt, 1).astype(np.float64)
    mu = S1 / n[:, None]
    C = S2 / n[:, None, None] - mu[:, :, None] * mu[:, None, :]
    cmax = np.abs(C).reshape(N, 9).max(1)
    ok = (cnt >= min_neighbors) & finite & np.isfinite(C).reshape(N, 9).all(1) & (cmax > 1e-12)
    ok &= np.trace(C, axis1=1, axis2=2) > 0
    ev = np.zeros((N, 3))
    if ok.any():
        ev[ok] = np.linalg.eigvalsh(C[ok])                           # ascending: e3, e2, e1
    e3, e2, e1 = ev[:, 0], ev[:, 1], ev[:, 2]
    with np.errstate(divide='ignore', invalid='ignore'):
        r21, r32 = e2 / e1, e3 / e2
        s = np.where(ok & (r21 < gamma_21) & (r32 < gamma_32), e3, 0.0)
        amb_s = near_s.copy()
        amb_s |= ok & (np.abs(r21 - gamma_21) <= RATIO_TOL * max(1.0, gamma_21))
        amb_s |= ok & (np.abs(r32 - gamma_32) <= RATIO_TOL * max(1.0, gamma_32))
        amb_s |= ok & (np.abs(e3) <= RATIO_TOL * np.abs(e1))
    amb_s |= (cnt >= min_neighbors) & finite & (np.abs(cmax - 1e-12) <= 1e-6 * 1e-12)

    # non-maximum suppression
    qi, pj, near_n = radius_pairs(X, F, tree, rnm)
    cnt_n = np.bincount(qi, minlength=N)
    beaten = np.zeros(N, bool)
    beaten[qi[s[pj] > s[qi]]] = True
    key = (s > 0) & (cnt_n >= min_neighbors) & ~beaten
    scale = np.maximum(np.abs(e1[qi]), np.abs(e1[pj]))
    tie = (np.abs(s[pj] - s[qi]) <= RATIO_TOL * scale) & (X64[pj] != X64[qi]).any(1) & ((s[pj] > 0) | (s[qi] > 0))
    amb = amb_s | near_n
    amb[qi[tie | amb_s[pj]]] = True
    return dict(idx=np.flatnonzero(key), saliency=s, e1=e1, amb=amb, radii=(rs, rnm), count_s=cnt, count_nm=cnt_n)


def iss_literal(X, salient_radius=0.0, non_max_radius=0.0, gamma_21=0.975, gamma_32=0.975, min_neighbors=5):
    """Open3D's ComputeISSKeypoints written out point by point (brute-force radius search with the kernel's distance,
    raw-cumulant covariance as utility::ComputeCovariance, IsLocalMaxima).  Small clouds only."""
    X = np.ascontiguousarray(X, np.float32)
    N = len(X)
    fin = np.isfinite(X).all(1)
    if salient_radius == 0 or non_max_radius == 0:
        tot, m = 0.0, 0
        for i in range(N):
            if not fin[i]:
                continue
            d = [float(fp32_dist(X[i:i + 1], X[j:j + 1])[0]) for j in range(N) if j != i and fin[j]]
            if d:
                tot += np.sqrt(min(d)); m += 1
        res = tot / m if m else 0.0
        salient_radius, non_max_radius = np.float32(6 * res), np.float32(4 * res)

    def search(i, r):
        r2 = np.float32(r) * np.float32(r)
        if not fin[i]:
            return []
        return [j for j in range(N) if fin[j] and fp32_dist(X[i:i + 1], X[j:j + 1])[0] < r2]

    third = np.zeros(N)
    for i in range(N):
        nb = search(i, salient_radius)
        if len(nb) < min_neighbors:
            continue
        P = X[nb].astype(np.float64)
        mean = P.sum(0) / len(nb)
        cov = (P.T @ P) / len(nb) - np.outer(mean, mean)
        if np.all(np.abs(cov) <= 1e-12) or not np.isfinite(cov).all():
            continue
        e = np.linalg.eigvalsh(cov)
        if e[1] / e[2] < gamma_21 and e[0] / e[1] < gamma_32:
            third[i] = e[0]
    kp = []
    for i in range(N):
        if third[i] > 0.0:
            nb = search(i, non_max_radius)
            if len(nb) >= min_neighbors and all(not third[i] < third[j] for j in nb):
                kp.append(i)
    return np.asarray(kp, np.int64), third
