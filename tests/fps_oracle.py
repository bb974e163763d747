"""Row f12 (SURVEY.md §8f): numpy fp64 replay of the farthest point sampling contract of include/ri_b200.h
(ri_furthest_point_sample_f32), vectorised over the points of a cloud.

    dist[i] = +inf for i < n;  s = 0
    for k in 0 .. m-1:  idx[k] = s;  dist = min(dist, (dx*dx + dy*dy) + dz*dz)  (fp64, dx = (double)x_i - (double)x_s)
                        s = first argmax of dist if its maximum is > 0, else s unchanged

numpy evaluates every operation in fp64 with round to nearest and never contracts, which is the kernel's arithmetic.
`dist = where(d < dist, d, dist)` keeps dist for NaN distances, as the contract's `d < dist[i] ? d : dist[i]` does."""
import numpy as np


def fps_one(xyz, n, m):
    """xyz [3, N] float32 (only the first n points are read) -> idx [m] int32."""
    if n == 0:
        return np.full(m, -1, np.int32)
    p = np.asarray(xyz, np.float32)[:, :n].astype(np.float64)
    dist = np.full(n, np.inf)
    out = np.empty(m, np.int32)
    s = 0
    with np.errstate(invalid="ignore", over="ignore"):
        for k in range(m):
            out[k] = s
            if k == m - 1:
                break
            d = p - p[:, s:s + 1]
            d = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
            dist = np.where(d < dist, d, dist)
            j = int(np.argmax(dist))               # first maximum; dist holds no NaN
            if dist[j] > 0.0:
                s = j
            else:                                  # every dist is 0: s never changes again
                out[k + 1:] = s
                break
    return out


def fps(xyz, m, lengths=None):
    """xyz [B, 3, N] float32, lengths [B] or None -> idx [B, m] int32."""
    xyz = np.asarray(xyz, np.float32)
    B, _, N = xyz.shape
    ns = [N] * B if lengths is None else [int(v) for v in lengths]
    return np.stack([fps_one(xyz[b], ns[b], m) for b in range(B)]) if B else np.zeros((0, m), np.int32)


def fps_literal(xyz, n, m):
    """The contract's loop word for word, one point at a time in Python floats (IEEE fp64) — for small clouds only."""
    if n == 0:
        return [-1] * m
    P = [[float(np.float32(xyz[c][i])) for c in range(3)] for i in range(n)]
    dist = [float("inf")] * n
    s, out = 0, []
    for _ in range(m):
        out.append(s)
        q = P[s]                                   # x_s: the point just taken (s moves during the loop)
        best = 0.0
        for i in range(n):
            dx, dy, dz = P[i][0] - q[0], P[i][1] - q[1], P[i][2] - q[2]
            d = (dx * dx + dy * dy) + dz * dz
            dist[i] = d if d < dist[i] else dist[i]
            if dist[i] > best:
                best = dist[i]
                s = i
    return out


# ---------------------------------------------------------------------------------------------- hand-made clouds
def collinear(n=17):
    x = np.arange(n, dtype=np.float32)
    return np.stack([x, 2 * x, -x]).astype(np.float32)


def lattice(k=4):
    """k^3 points of an integer lattice: every distance is an exact small integer, so ties are everywhere."""
    g = np.stack(np.meshgrid(*[np.arange(k)] * 3, indexing="ij"), 0).reshape(3, -1)
    return g.astype(np.float32)


def duplicates(seed=0, n=24):
    """Random points, each written three times (in a shuffled order)."""
    rng = np.random.default_rng(seed)
    p = rng.standard_normal((3, n // 3)).astype(np.float32)
    p = np.concatenate([p, p, p], 1)
    return p[:, rng.permutation(p.shape[1])].copy()


def identical(n=9):
    return np.tile(np.array([[0.5], [-1.25], [3.0]], np.float32), (1, n))


def with_nan(seed=1, n=20, at=7):
    rng = np.random.default_rng(seed)
    p = rng.standard_normal((3, n)).astype(np.float32)
    p[1, at] = np.nan
    return p


HAND_MADE = {"collinear": collinear, "lattice": lattice, "duplicates": duplicates, "identical": identical,
             "nan": with_nan}
