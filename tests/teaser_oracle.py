"""fp64 replay of csrc/teaser.cu (row f10, TEASER++ with a known scale) for the tests and tools only, one pair at a time.

    graph     edge (i, j), i != j, iff |l_a(i,j) - l_b(i,j)| <= beta, beta = 2 * noise_bound * sqrt(cbar2); l = |u - v| in
              fp64 from the fp32 coordinates as sqrt((dx*dx + dy*dy) + dz*dz).  numpy rounds every operation and never
              contracts, so the graph is the kernel's bit for bit.
    order     pi sorts the vertices by degree descending, then index ascending.  Vertices are relabelled by their rank
              in pi, and bitsets are Python integers in rank space: "first in pi order" is the lowest set bit.
    clique    heuristic incumbent from the first min(M, 64) ranks, peeling below |best|, then the BBMC branch and bound
              (greedy colouring in rank order, vertices visited in reverse colouring order, prune on |C| + colour <= |best|)
              with one node per expand call and a budget of max_clique_nodes calls.  This is the clique bit for bit.
    rotation  GNC-TLS over the chain TIMs of the sorted clique; Horn's rotation from the largest eigenvector of its 4x4
              matrix (numpy eigh; the kernel runs Jacobi sweeps).  `replay` reports the gap between the two largest
              eigenvalues of every solve and the smallest relative distance of a residual to a weight threshold, so a
              fixture can be shown to be well conditioned before the GPU pose is compared with it.
    voting    per axis, the consensus sets of the sweep over the interval endpoints x_k -/+ r, estimate = their mean,
              cost = sum_in (x - mean)^2 + |out| r^2; the minimum cost, the earliest event on ties.
The product package never imports this module.
"""
from dataclasses import dataclass, field

import numpy as np

HEURISTIC_STARTS = 64


def f32(v):
    return float(np.float32(v))


def edge_lengths(x, rows, cols):
    """[len(rows), len(cols)] fp64 |x_r - x_c| in the kernel's operation order (x fp32 [M,3])."""
    x = np.asarray(x, np.float32).astype(np.float64)
    d = x[rows][:, None, :] - x[cols][None, :, :]
    return np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])


def beta_of(noise_bound, cbar2):
    return 2.0 * f32(noise_bound) * np.sqrt(f32(cbar2))


def adjacency(a, b, beta, order=None, chunk=512):
    """bool [M, M] consistency graph; with `order` (rank -> vertex) relabelled into rank space."""
    M = len(a)
    order = np.arange(M) if order is None else np.asarray(order)
    out = np.zeros((M, M), bool)
    for s in range(0, M, chunk):
        r = order[s:s + chunk]
        e = np.abs(edge_lengths(a, r, order) - edge_lengths(b, r, order)) <= beta
        e[np.arange(len(r)), np.arange(s, s + len(r))] = False
        out[s:s + chunk] = e
    return out


def degrees(a, b, beta, chunk=512):
    M = len(a)
    deg = np.zeros(M, np.int64)
    for s in range(0, M, chunk):
        r = np.arange(s, min(s + chunk, M))
        e = np.abs(edge_lengths(a, r, np.arange(M)) - edge_lengths(b, r, np.arange(M))) <= beta
        e[np.arange(len(r)), r] = False
        deg[r] = e.sum(1)
    return deg


def pi_order(deg):
    """rank -> vertex: degree descending, then index ascending."""
    return np.lexsort((np.arange(len(deg)), -np.asarray(deg)))


def bit_rows(adj):
    """bool [M, M] -> list of Python ints, bit c of row r = adj[r, c]."""
    packed = np.packbits(adj, axis=1, bitorder='little')
    return [int.from_bytes(row.tobytes(), 'little') for row in packed]


def low(x):
    return (x & -x).bit_length() - 1


def bits(x):
    out = []
    while x:
        v = low(x)
        out.append(v)
        x &= x - 1
    return out


def greedy_clique(rows, s):
    """The heuristic clique from rank s: C = {s}, cand = N(s); add the lowest rank of cand, cand &= its neighbourhood."""
    C, cand = [s], rows[s]
    while cand:
        u = low(cand)
        C.append(u)
        cand &= rows[u]
    return C


def colour(rows, P):
    """BBMC greedy colouring of P in rank order -> [(vertex, colour)] in colouring order."""
    out, U, k = [], P, 0
    while U:
        k += 1
        Q = U
        while Q:
            v = low(Q)
            out.append((v, k))
            U &= ~(1 << v)
            Q &= ~rows[v] & ~(1 << v)
    return out


@dataclass
class Clique:
    ranks: list                      # the clique in rank space, in the order found
    exact: bool
    nodes: int                       # expand calls made
    heuristic: int                   # size of the incumbent before the exact search
    alive: int                       # vertices left by the peeling


def max_clique(rows, max_nodes):
    """The kernel's search over the rank-space rows (a list of M Python ints)."""
    M = len(rows)
    best = []
    for s in range(min(M, HEURISTIC_STARTS)):
        C = greedy_clique(rows, s)
        if len(C) > len(best):
            best = C
    heuristic = len(best)
    alive = (1 << M) - 1
    while True:
        dead = 0
        for v in bits(alive):
            if (rows[v] & alive).bit_count() < len(best):
                dead |= 1 << v
        if not dead:
            break
        alive &= ~dead
    nodes, exact = 0, True

    class Stop(Exception):
        pass

    def expand(C, P):
        nonlocal nodes, best
        if nodes == max_nodes:
            raise Stop
        nodes += 1
        order = colour(rows, P)
        for v, c in reversed(order):
            if len(C) + c <= len(best):
                return
            NP = P & rows[v]
            if NP == 0:
                if len(C) + 1 > len(best):
                    best = C + [v]
            else:
                expand(C + [v], NP)
            P &= ~(1 << v)

    import sys
    limit = sys.getrecursionlimit()
    sys.setrecursionlimit(max(limit, 4 * M + 1000))
    try:
        expand([], alive)
    except Stop:
        exact = False
    finally:
        sys.setrecursionlimit(limit)
    return Clique(best, exact, nodes, heuristic, alive.bit_count())


def clique_of(a, b, noise_bound, cbar2=1.0, max_clique_nodes=1 << 20):
    """-> (clique as ascending match positions [K] int64, Clique record)."""
    a = np.asarray(a, np.float32); b = np.asarray(b, np.float32)
    M = len(a)
    if M == 0:
        return np.zeros(0, np.int64), Clique([], True, 0, 0, 0)
    beta = beta_of(noise_bound, cbar2)
    order = pi_order(degrees(a, b, beta))
    rows = bit_rows(adjacency(a, b, beta, order))
    c = max_clique(rows, int(max_clique_nodes))
    return np.sort(order[np.asarray(c.ranks, np.int64)]), c


# ---------------------------------------------------------------------------------------------- rotation, translation
def horn(S):
    """Horn's rotation from S = sum w v w^T (maps v onto w) -> (R [3,3], gap between the two largest eigenvalues)."""
    Sxx, Sxy, Sxz, Syx, Syy, Syz, Szx, Szy, Szz = np.asarray(S).reshape(9)
    N = np.array([[Sxx + Syy + Szz, Syz - Szy, Szx - Sxz, Sxy - Syx],
                  [Syz - Szy, Sxx - Syy - Szz, Sxy + Syx, Szx + Sxz],
                  [Szx - Sxz, Sxy + Syx, -Sxx + Syy - Szz, Syz + Szy],
                  [Sxy - Syx, Szx + Sxz, Syz + Szy, -Sxx - Syy + Szz]])
    ev, V = np.linalg.eigh(N)
    qw, qx, qy, qz = V[:, 3] / np.linalg.norm(V[:, 3])
    R = np.array([[1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw)],
                  [2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw)],
                  [2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)]])
    return R, float(ev[3] - ev[2])


@dataclass
class Gnc:
    R: np.ndarray
    iterations: int
    gaps: list = field(default_factory=list)       # eigen gap of Horn's matrix per solve
    margins: list = field(default_factory=list)    # per iteration: smallest |r2 - th| / th over both weight thresholds


def gnc_tls(v, w, c2, gnc_factor=1.4, max_iterations=100, cost_threshold=1e-12):
    """TEASER++'s GNC-TLS rotation over TIM pairs v, w [K,3] fp64 (w ~ R v) with bound^2 = c2."""
    K = len(v)
    wt = np.ones(K)
    R = np.eye(3)
    out = Gnc(R, 0)
    mu, prev = 1.0, 0.0
    for it in range(max_iterations):
        S = (v * wt[:, None]).T @ w
        R, gap = horn(S)
        out.gaps.append(gap)
        out.iterations = it + 1
        d = w - v @ R.T
        r2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        if it == 0:
            mu = 1.0 / (2.0 * r2.max() / c2 - 1.0)
            if mu <= 0:
                break
        th1 = (mu + 1) / mu * c2
        th2 = mu / (mu + 1) * c2
        out.margins.append(float(min(np.abs(r2 - th1).min() / th1, np.abs(r2 - th2).min() / th2)))
        cost = float(np.sum(wt * r2))
        wt = np.where(r2 >= th1, 0.0, np.where(r2 <= th2, 1.0, np.sqrt(c2 * mu * (mu + 1) / np.maximum(r2, 1e-300)) - mu))
        diff = abs(cost - prev)
        mu *= gnc_factor
        prev = cost
        if diff < cost_threshold:
            break
    out.R = R
    return out


def events(x, r):
    """The sweep's events in order: [(value, type (0 enter, 1 leave), index)]."""
    ev = [(float(xi - r), 0, i) for i, xi in enumerate(x)] + [(float(xi + r), 1, i) for i, xi in enumerate(x)]
    return sorted(ev)


def adaptive_voting(x, r):
    """TEASER++'s ScalarTLSEstimator with equal ranges r: -> (estimate, cost, consensus mask)."""
    x = np.asarray(x, np.float64)
    K = len(x)
    inside = np.zeros(K, bool)
    best = None
    for val, typ, i in events(x, r):
        inside[i] = typ == 0
        n = int(inside.sum())
        if n == 0:
            continue
        xs = x[inside]
        est = xs.sum() / n
        cost = float(np.sum((xs - est) ** 2) + (K - n) * r * r)
        if best is None or cost < best[1]:
            best = (est, cost, inside.copy())
    return best


def tls_cost(x, r, t):
    """The truncated least squares cost sum min((x - t)^2, r^2) of a translation component t."""
    return np.minimum((np.asarray(x, np.float64) - t) ** 2, r * r).sum()


# ---------------------------------------------------------------------------------------------- the whole pair
@dataclass
class Replay:
    clique: np.ndarray               # ascending match positions
    exact: bool
    posed: bool
    T: np.ndarray                    # [4,4] fp64 src -> tgt (identity without a pose)
    T32: np.ndarray
    inliers: int
    search: Clique = None
    gnc: Gnc = None


def replay(a, b, noise_bound, cbar2=1.0, gnc_factor=1.4, max_iterations=100, cost_threshold=1e-12,
           max_clique_nodes=1 << 20, inlier_dist=None):
    """The kernel's result for one pair of matched coordinates a, b [M,3] (src[idx1[:M]], tgt[idx2[:M]]).  Float
    arguments are rounded to fp32, as the C ABI takes them."""
    nb, c2f = f32(noise_bound), f32(cbar2)
    inlier_dist = f32(nb if inlier_dist is None else inlier_dist)
    a32 = np.asarray(a, np.float32); b32 = np.asarray(b, np.float32)
    clique, search = clique_of(a32, b32, nb, c2f, max_clique_nodes)
    eye = np.eye(4)
    if len(a32) < 3 or len(clique) < 3:
        return Replay(clique, search.exact, False, eye, eye.astype(np.float32), 0, search)
    A = a32[clique].astype(np.float64); B = b32[clique].astype(np.float64)
    nxt = np.roll(np.arange(len(clique)), -1)
    beta = beta_of(nb, c2f)
    g = gnc_tls(A[nxt] - A, B[nxt] - B, beta * beta, f32(gnc_factor), int(max_iterations), f32(cost_threshold))
    X = B - A @ g.R.T
    rng = nb * np.sqrt(c2f)
    t = np.array([adaptive_voting(X[:, k], rng)[0] for k in range(3)])
    T = np.eye(4)
    T[:3, :3] = g.R
    T[:3, 3] = t
    T32 = T.astype(np.float32)
    return Replay(clique, search.exact, True, T, T32, count_inliers(T32, a32, b32, inlier_dist), search, g)


def count_inliers(T, a, b, dist):
    """Matches within dist under T, in fp64 (the kernel's fp32 count may differ on residuals at the threshold)."""
    T = np.asarray(T, np.float64)
    d = np.asarray(a, np.float64) @ T[:3, :3].T + T[:3, 3] - np.asarray(b, np.float64)
    return int((np.linalg.norm(d, axis=1) < dist).sum())
