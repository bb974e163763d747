"""CPU reference of FPFH descriptors (row f8), for the tests and tools/bench_fpfh.py only.

Open3D's compute_fpfh_feature (pipelines/registration/Feature.cpp: ComputePairFeatures, ComputeSPFHFeature,
ComputeFPFHFeature) restated in numpy fp64 on given neighbour lists, with the rules of csrc/fpfh.cu (include/ri_b200.h,
ri_compute_fpfh_f32): every fp64 operation is rounded on its own, in the kernel's order, so only acos / atan2 (glibc here,
libdevice there) can differ.  Where that difference could move a bin the bin is flagged ambiguous:
    the pre-floor bin value is within 1e-9 of an integer, or 0 < ||a1| - |a2|| < 1e-12 at the swap test.
Also a brute-force builder of the hybrid neighbour lists with the fp32 fma-chain distance emulated exactly.
Clouds are point-major [N,3] here.  The product package never imports this module.
"""
import numpy as np

AMBIG_BIN = 1e-9
AMBIG_SWAP = 1e-12


def _dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1],
                     a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], -1)


def pair_features(p1, n1, p2, n2, swap_tol=AMBIG_SWAP):
    """Arrays [...,3] (fp32 values) -> (f [...,3] fp64 = (f0, f1, f2), swap_ambiguous [...] bool)."""
    p1, n1, p2, n2 = (np.asarray(a, np.float64) for a in (p1, n1, p2, n2))
    dp = p2 - p1
    L = np.sqrt(_dot(dp, dp))
    with np.errstate(divide='ignore', invalid='ignore'):
        a1 = _dot(n1, dp) / L
        a2 = _dot(n2, dp) / L
        swap = np.arccos(np.abs(a1)) > np.arccos(np.abs(a2))
        gap = np.abs(np.abs(a1) - np.abs(a2))
        amb = (gap != 0) & (gap < swap_tol)             # equal |a1|, |a2| (equal normals) compare equal anywhere
    u = np.where(swap[..., None], n2, n1)
    s = np.where(swap[..., None], n1, n2)
    dp = np.where(swap[..., None], -dp, dp)
    f2 = np.where(swap, -a2, a1)
    v = _cross(dp, u)
    vn = np.sqrt(_dot(v, v))
    with np.errstate(divide='ignore', invalid='ignore'):
        v = v / vn[..., None]
    w = _cross(u, v)
    f1 = _dot(v, s)
    f0 = np.arctan2(_dot(w, s), _dot(u, s))
    zero = (L == 0) | (vn == 0)
    f = np.stack([f0, f1, f2], -1)
    f[zero] = 0.0
    return f, amb & ~(L == 0)


def bin_values(f):
    """f [...,3] -> the pre-floor bin values [...,3]: 11 (f0 + pi) / (2 pi), 11 (f1 + 1) * 0.5, 11 (f2 + 1) * 0.5."""
    return np.stack([11.0 * (f[..., 0] + np.pi) / (2.0 * np.pi), 11.0 * (f[..., 1] + 1.0) * 0.5,
                     11.0 * (f[..., 2] + 1.0) * 0.5], -1)


def bins(f, bin_tol=AMBIG_BIN):
    """-> (bins [...,3] int in [0, 10], ambiguous [...,3] bool)."""
    x = bin_values(f)
    with np.errstate(invalid='ignore'):
        b = np.clip(np.floor(x), 0, 10).astype(np.int64)
        amb = np.abs(x - np.rint(x)) < bin_tol
    return b, amb


def spfh_counts(xyz, normals, idx, count, bin_tol=AMBIG_BIN, swap_tol=AMBIG_SWAP):
    """xyz, normals [N,3]; idx [N,K] neighbour lists, the first count[i] of row i used
    -> (counts [N,33] int64, ambiguous [N] bool: some pair of the point has an ambiguous bin or swap test).
    Wider tolerances serve comparisons across inputs that differ by rounding (a rotated copy)."""
    xyz = np.asarray(xyz, np.float32); normals = np.asarray(normals, np.float32)
    idx = np.asarray(idx, np.int64); count = np.asarray(count, np.int64)
    N, K = idx.shape
    c = np.zeros((N, 33), np.int64)
    amb = np.zeros(N, bool)
    if K < 2:
        return c, amb
    j = np.clip(idx[:, 1:], 0, max(N - 1, 0))
    use = np.arange(1, K)[None, :] < count[:, None]
    f, samb = pair_features(xyz[:, None, :], normals[:, None, :], xyz[j], normals[j], swap_tol)
    b, bamb = bins(f, bin_tol)
    amb = ((samb | bamb.any(-1)) & use).any(1)
    rows = np.broadcast_to(np.arange(N)[:, None], use.shape)[use]
    for g in range(3):
        np.add.at(c, (rows, 11 * g + b[..., g][use]), 1)
    return c, amb


def spfh_from_counts(c, count):
    """counts [N,33], list lengths [N] -> spfh [N,33] fp64 = c * (100 / (n - 1)), zeros for n <= 1."""
    count = np.asarray(count, np.int64)
    with np.errstate(divide='ignore'):
        incr = np.where(count > 1, 100.0 / (count - 1).astype(np.float64), 0.0)
    return np.asarray(c, np.float64) * incr[:, None]


def fpfh_from_spfh(xyz, spfh, idx, count):
    """Open3D's ComputeFPFHFeature on given lists: -> fpfh [N,33] fp64, sequential in list order."""
    xyz = np.asarray(xyz, np.float32).astype(np.float64)
    idx = np.asarray(idx, np.int64); count = np.asarray(count, np.int64)
    N, K = idx.shape
    feat = np.zeros((N, 33)); s = np.zeros((N, 3))
    for k in range(1, K):
        use = k < count
        j = np.clip(idx[:, k], 0, max(N - 1, 0))
        d = xyz[j] - xyz
        w = _dot(d, d)
        use &= w != 0
        with np.errstate(divide='ignore', invalid='ignore'):
            val = spfh[j] / w[:, None]
        val[~use] = 0.0
        feat += val
        for g in range(3):                               # Open3D adds val to sum[j / 11] one j at a time
            for jj in range(11 * g, 11 * g + 11):
                s[:, g] += val[:, jj]
    with np.errstate(divide='ignore'):
        scale = np.where(s != 0, 100.0 / np.where(s != 0, s, 1.0), 0.0)
    out = feat * np.repeat(scale, 11, axis=1) + spfh
    out[count <= 1] = 0.0
    return out


def compute_fpfh(xyz, normals, idx, count):
    """-> (fpfh [N,33] fp64, spfh [N,33] fp64, counts [N,33] int, ambiguous [N] bool) on given lists."""
    c, amb = spfh_counts(xyz, normals, idx, count)
    spfh = spfh_from_counts(c, count)
    return fpfh_from_spfh(xyz, spfh, idx, count), spfh, c, amb


# ---------------------------------------------------------------------------------------------- neighbour lists
def _fma32(a, b, c):
    """fp32 fma(a, b, c) rounded once: a*b is exact in fp64, the sum's fp64 rounding error is recovered (TwoSum) and used
    to settle a result that lands on an fp32 rounding midpoint."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c = c.astype(np.float64)
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)                        # s + e == p + c exactly
    r = s.astype(np.float32)
    rd = s - r.astype(np.float64)
    other = np.nextafter(r, np.where(rd > 0, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
    mid = (rd != 0) & (np.abs(other.astype(np.float64) - s) == np.abs(rd))
    beyond = mid & (e != 0) & (np.sign(e) == np.sign(rd))  # the true value is past the midpoint, on `other`'s side
    return np.where(beyond, other, r)


def fp32_dist(q, p):
    """fma(dz,dz, fma(dy,dy, dx*dx)) in fp32 with d* = q - p: q [...,3], p [...,3] fp32."""
    d = np.asarray(q, np.float32) - np.asarray(p, np.float32)
    dx, dy, dz = d[..., 0], d[..., 1], d[..., 2]
    return _fma32(dz, dz, _fma32(dy, dy, dx * dx))


def hybrid_lists(xyz, radius, max_nn):
    """Brute force: each point's max_nn smallest (d, index) with d < min(radius^2 in fp32, 10000).
    -> (idx [N,max_nn] int64, -1 beyond count; count [N])."""
    xyz = np.asarray(xyz, np.float32)
    N = len(xyz)
    r = np.float32(radius)
    lim = min(np.float32(r * r), np.float32(10000.0))
    idx = np.full((N, max_nn), -1, np.int64)
    count = np.zeros(N, np.int64)
    for i in range(N):
        d = fp32_dist(xyz[i][None], xyz)
        order = np.lexsort((np.arange(N), d))
        order = order[d[order] < lim][:max_nn]
        idx[i, :len(order)] = order
        count[i] = len(order)
    return idx, count
