"""fp64 replay of csrc/fgr.cu (row f7, Open3D's Fast Global Registration) for the tests and tools only, one pair at a time.

    tuple test   trial t of pair p: r0 = mix64(seed ^ (p << 32) ^ (uint32)t), r1 = mix64(r0), r2 = mix64(r1), i_k = r_k % M
                 (pose_oracle.mix64, bit for bit); edge lengths sqrt((dx*dx + dy*dy) + dz*dz) in fp64 from the fp32
                 coordinates, accepted when l_a * s < l_b < l_a / s on all three edges.  numpy rounds every operation and never
                 contracts, so the list is the kernel's bit for bit.  The first max_tuples accepted trials, in trial order.
    normalise    means of all points, scale = the largest centred norm; points used as (x - mu) * (1 / g).
    GNC          `iterations` Gauss-Newton steps on J^T W J x = -J^T W r (numpy cholesky / solve), T' = Delta T'.
    output       inverse of [R' | mu_s - R' mu_t + g t'], and the inlier count under its fp32 rounding.
The GNC loop is the kernel's up to summation order; `replay` also reports the smallest eigenvalue of J^T W J at every
iteration, so a fixture can be shown to be well conditioned before the GPU result is compared with it.
The product package never imports this module.
"""
from dataclasses import dataclass, field

import numpy as np

from pose_oracle import MASK64, mix64

MIN_CORR = 10


def trial_indices(seed, pair, M, trials):
    """[T, 3] int64 match positions of the trials in `trials` (an int array) of pair `pair` with M matches."""
    t = np.asarray(trials, np.int64)
    key = (int(seed) & MASK64) ^ ((int(pair) & MASK64) << 32 & MASK64)
    r0 = mix64(np.uint64(key) ^ t.astype(np.uint32).astype(np.uint64))
    r1 = mix64(r0)
    r2 = mix64(r1)
    return np.stack([(r % np.uint64(M)).astype(np.int64) for r in (r0, r1, r2)], -1)


def _edges(x, idx):
    """[T, 3] fp64 edge lengths |x_i0 - x_i1|, |x_i1 - x_i2|, |x_i2 - x_i0|, in the kernel's operation order."""
    x = np.asarray(x, np.float32).astype(np.float64)
    out = []
    for i, j in ((0, 1), (1, 2), (2, 0)):
        d = x[idx[:, i]] - x[idx[:, j]]
        out.append(np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]))
    return np.stack(out, -1)


def tuple_accept(a, b, idx, tuple_scale):
    """[T] bool: the kernel's edge test of the trials idx [T, 3] on matched coordinates a, b [M, 3] (fp32)."""
    s = float(np.float32(tuple_scale))
    la, lb = _edges(a, idx), _edges(b, idx)
    return np.all((la * s < lb) & (lb < la / s), axis=1)


def tuple_list(a, b, seed, pair, tuple_scale=0.95, max_tuples=1000, chunk=65536):
    """The correspondence list of the tuple test: [3 * accepted] int64 match positions."""
    M = len(a)
    if M < 3:
        return np.zeros(0, np.int64)
    trials = 100 * M
    out, n = [], 0
    for base in range(0, trials, chunk):
        idx = trial_indices(seed, pair, M, np.arange(base, min(base + chunk, trials)))
        ok = idx[tuple_accept(a, b, idx, tuple_scale)]
        out.append(ok[:max_tuples - n])
        n += len(out[-1])
        if n >= max_tuples:
            break
    return np.concatenate(out).reshape(-1) if out else np.zeros(0, np.int64)


def euler_zyx(x0, x1, x2):
    """Rz(x2) Ry(x1) Rx(x0)."""
    ca, sa, cb, sb, cg, sg = np.cos(x0), np.sin(x0), np.cos(x1), np.sin(x1), np.cos(x2), np.sin(x2)
    return np.array([[cg * cb, cg * sb * sa - sg * ca, cg * sb * ca + sg * sa],
                     [sg * cb, sg * sb * sa + cg * ca, sg * sb * ca - cg * sa],
                     [-sb, cb * sa, cb * ca]])


def normal_equations(p, qh, Tp, par):
    """J^T W J [6,6] and J^T W r [6] of the correspondences p [L,3] (normalised source) and qh [L,3] (normalised target)
    under T' [4,4]: r = p - T' qh, w = (par / (r.r + par))^2."""
    q = qh @ Tp[:3, :3].T + Tp[:3, 3]
    r = p - q
    w = (par / (np.sum(r * r, 1) + par)) ** 2
    L = len(p)
    J = np.zeros((L, 3, 6))
    J[:, 0, 1], J[:, 0, 2], J[:, 0, 3] = -q[:, 2], q[:, 1], -1.0
    J[:, 1, 0], J[:, 1, 2], J[:, 1, 4] = q[:, 2], -q[:, 0], -1.0
    J[:, 2, 0], J[:, 2, 1], J[:, 2, 5] = -q[:, 1], q[:, 0], -1.0
    JTJ = np.einsum('l,lki,lkj->ij', w, J, J)
    JTr = np.einsum('l,lki,lk->i', w, J, r)
    return JTJ, JTr


def gn_step(JTJ, JTr):
    """x = -(J^T J)^-1 J^T r by Cholesky, or None where the kernel keeps Delta = I (not positive definite, not finite)."""
    try:
        C = np.linalg.cholesky(JTJ)
    except np.linalg.LinAlgError:
        return None
    x = -np.linalg.solve(C.T, np.linalg.solve(C, JTr))
    return x if np.all(np.isfinite(x)) else None


def delta(x):
    D = np.eye(4)
    D[:3, :3] = euler_zyx(x[0], x[1], x[2])
    D[:3, 3] = x[3:]
    return D


@dataclass
class Replay:
    corr: np.ndarray                 # the list's match positions
    posed: bool
    T: np.ndarray                    # [4,4] fp64 src -> tgt (identity without a pose)
    T32: np.ndarray                  # its fp32 rounding, what the kernel returns
    inliers: int                     # count under T32 (0 without a pose)
    min_eig: list = field(default_factory=list)    # smallest eigenvalue of J^T W J per iteration
    solved: list = field(default_factory=list)     # per iteration: the step was applied


def replay(src, tgt, a, b, seed=0, pair=0, max_corr_dist=0.025, iterations=64, division_factor=1.4,
           use_absolute_scale=False, decrease_mu=True, tuple_test=True, tuple_scale=0.95, max_tuples=1000,
           inlier_dist=None):
    """The kernel's result for one pair: src [n1,3], tgt [n2,3] the clouds (for the normalisation), a, b [M,3] the matched
    coordinates (src[idx1[:M]], tgt[idx2[:M]]).  Float arguments are rounded to fp32, as the C ABI takes them."""
    f = lambda v: float(np.float32(v))
    max_corr_dist, division_factor = f(max_corr_dist), f(division_factor)
    inlier_dist = f(max_corr_dist if inlier_dist is None else inlier_dist)
    a32 = np.asarray(a, np.float32); b32 = np.asarray(b, np.float32)
    M = len(a32)
    corr = tuple_list(a32, b32, seed, pair, tuple_scale, max_tuples) if tuple_test else np.arange(M)
    eye = np.eye(4)
    if M < 3 or len(corr) < MIN_CORR:
        return Replay(corr, False, eye, eye.astype(np.float32), 0)
    S = np.asarray(src, np.float32).astype(np.float64); G = np.asarray(tgt, np.float32).astype(np.float64)
    mu_s, mu_t = S.mean(0), G.mean(0)
    scale = np.sqrt(max(np.max(np.sum((S - mu_s) ** 2, 1)), np.max(np.sum((G - mu_t) ** 2, 1))))
    g, par = (1.0, scale) if use_absolute_scale else (scale, 1.0)
    ig = 1.0 / g
    p = (a32[corr].astype(np.float64) - mu_s) * ig
    qh = (b32[corr].astype(np.float64) - mu_t) * ig
    Tp = np.eye(4)
    r = Replay(corr, True, eye, eye, 0)
    for it in range(iterations):
        if decrease_mu and it % 4 == 0 and par > max_corr_dist:
            par /= division_factor
        JTJ, JTr = normal_equations(p, qh, Tp, par)
        r.min_eig.append(float(np.linalg.eigvalsh(JTJ)[0]))
        x = gn_step(JTJ, JTr)
        r.solved.append(x is not None)
        if x is not None:
            Tp = delta(x) @ Tp
    T_ts = np.eye(4)
    T_ts[:3, :3] = Tp[:3, :3]
    T_ts[:3, 3] = mu_s - Tp[:3, :3] @ mu_t + g * Tp[:3, 3]
    r.T = np.eye(4)
    r.T[:3, :3] = Tp[:3, :3].T
    r.T[:3, 3] = -Tp[:3, :3].T @ T_ts[:3, 3]
    r.T32 = r.T.astype(np.float32)
    r.inliers = count_inliers(r.T32, a32, b32, inlier_dist)
    return r


def count_inliers(T, a, b, dist):
    """Matches within dist under T, in fp64 (the kernel's fp32 count may differ on residuals at the threshold)."""
    T = np.asarray(T, np.float64)
    d = np.asarray(a, np.float64) @ T[:3, :3].T + T[:3, 3] - np.asarray(b, np.float64)
    return int((np.linalg.norm(d, axis=1) < dist).sum())
