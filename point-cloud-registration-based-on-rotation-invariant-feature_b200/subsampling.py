"""Barycentre grid subsampling on the GPU — the reference's `utils/grid_subsampleing.py:3-21` API over csrc/gridsub.cu
(reference implementation: a CPU CPython extension, cpp_wrappers/cpp_subsampling/grid_subsampling/grid_subsampling.cpp).

`grid_sub_sampling(points, features=None, labels=None, grid_size=0.1, verbose=0)` keeps the reference's signature and its
return convention (points; points, features; points, labels; or all three — `wrapper.cpp:265-284`).  numpy inputs come back
as numpy arrays (the reference's types), CUDA tensors come back as CUDA tensors.  Cells are returned in ascending cell
index (the reference: unordered_map order), barycentres and mean features are bit-identical to the reference's.

`farthest_point_batch(clouds, num_samples)` turns the variable-length output of `grid_sub_sampling_many` into one fixed-size
batch by farthest point sampling (csrc/fps.cu).
"""
import numpy as np
import torch

from .backend import _backend


def _prepare(points, features, labels, dev):
    """Device tensors of one cloud in the shapes the op takes, with the reference wrapper's shape errors."""
    pts = torch.as_tensor(points, dtype=torch.float32).to(dev).contiguous()
    if pts.dim() != 2 or pts.shape[1] != 3:
        raise RuntimeError("Wrong dimensions : points.shape is not (N, 3)")                      # wrapper.cpp:118-125
    N = pts.shape[0]
    if features is None:
        f = torch.empty((N, 0), dtype=torch.float32, device=dev)
    else:
        f = torch.as_tensor(features, dtype=torch.float32).to(dev).contiguous()
        if f.dim() != 2 or f.shape[0] != N:
            raise RuntimeError("Wrong dimensions : features.shape is not (N, d)")                # wrapper.cpp:127-145
    if labels is None:
        l = torch.empty((N, 0), dtype=torch.int32, device=dev)
    else:
        l = torch.as_tensor(labels).to(torch.int32).to(dev).contiguous()
        if l.dim() > 2 or l.shape[0] != N:
            raise RuntimeError("Wrong dimensions : classes.shape is not (N,) or (N, d)")         # wrapper.cpp:147-162
        l = l.reshape(N, -1)
    return pts, f, l


def grid_sub_sampling_many(clouds, grid_size=0.1, device=None):
    """Several scans in one go: `clouds` is a list of `points` or `(points, features)` or `(points, features, labels)` (CUDA
    tensors or numpy arrays; features / labels may be None).  Every scan's kernels are enqueued back to back and the output
    lengths are read with ONE host synchronisation at the end (the single-cloud call reads its length after every scan, which
    leaves the GPU idle while the host prepares the next one).  Returns a list of tuples (points, features, labels) of CUDA
    tensors, None where the input had none; results identical to grid_sub_sampling()."""
    items = [c if isinstance(c, (tuple, list)) else (c,) for c in clouds]
    items = [tuple(c) + (None,) * (3 - len(c)) for c in items]
    if not items:
        return []
    first = items[0][0]
    dev = torch.device(device) if device is not None else (first.device if isinstance(first, torch.Tensor) else torch.device("cuda"))
    if dev.type != "cuda":
        raise RuntimeError("grid_sub_sampling runs on a CUDA device only (no CPU path exists in this package)")
    raw = []
    for (p, f, l) in items:
        pts, ft, lb = _prepare(p, f, l, dev)
        raw.append(torch.ops.ri.grid_subsample(pts, ft, lb, float(grid_size)) + (f is not None, l is not None))
    counts = torch.cat([r[3] for r in raw]).cpu().tolist()        # the only host synchronisation
    return [(op[:M], of[:M] if has_f else None, ol[:M] if has_l else None) for (op, of, ol, _, has_f, has_l), M in zip(raw, counts)]


def grid_sub_sampling(points, features=None, labels=None, grid_size=0.1, verbose=0, device=None):
    as_numpy = not isinstance(points, torch.Tensor)
    dev = torch.device(device) if device is not None else (torch.device("cuda") if as_numpy else points.device)
    if dev.type != "cuda":
        raise RuntimeError("grid_sub_sampling runs on a CUDA device only (no CPU path exists in this package)")
    pts, f, l = _prepare(points, features, labels, dev)
    op, of, ol, cnt = torch.ops.ri.grid_subsample(pts, f, l, float(grid_size))
    M = int(cnt.item())                                       # the only host synchronisation: the output length
    out = [op[:M]]
    if features is not None:
        out.append(of[:M])
    if labels is not None:
        out.append(ol[:M])
    if as_numpy:
        out = [o.cpu().numpy() for o in out]
    return out[0] if len(out) == 1 else tuple(out)


def farthest_point_batch(clouds, num_samples):
    """Variable-length clouds -> one fixed-size batch by farthest point sampling (csrc/fps.cu), the bridge from
    grid_sub_sampling_many to the batched ops that take dense [B, N, 3] clouds (normals, FPFH, registration).

    `clouds` is a list of CUDA point tensors [n_b, 3] or of tuples (points, features, ...) as grid_sub_sampling_many
    returns them (features [n_b, C] or None; further entries are ignored).  The clouds are padded into one [B, 3, N_max]
    batch; their lengths are known on the host, so nothing waits for the GPU.  Each cloud is sampled from its own first
    point, covering the whole cloud rather than a prefix of it.  A cloud with fewer than num_samples distinct points
    repeats its last pick; an empty cloud gives idx -1 and undefined rows.

    Returns (points [B, m, 3], features [B, m, C] or None, idx [B, m] int32), m = num_samples, rows in sampling order.
    Features are gathered only when every cloud has them (with one channel count)."""
    items = [c if isinstance(c, (tuple, list)) else (c,) for c in clouds]
    if not items:
        raise ValueError("farthest_point_batch needs at least one cloud")
    pts = [torch.as_tensor(c[0]) for c in items]
    feats = [c[1] if len(c) > 1 else None for c in items]
    dev = pts[0].device
    if dev.type != "cuda":
        raise RuntimeError("farthest_point_batch runs on a CUDA device only (no CPU path exists in this package)")
    for p in pts:
        if p.dim() != 2 or p.shape[1] != 3 or p.device != dev:
            raise RuntimeError("every cloud must be a [n, 3] tensor on %s" % dev)
    has_f = all(f is not None for f in feats)
    if not has_f and any(f is not None for f in feats):
        raise ValueError("either every cloud has features or none has")
    lengths = [int(p.shape[0]) for p in pts]
    B, N = len(pts), max(lengths)
    xyz = torch.zeros((B, 3, N), dtype=torch.float32, device=dev)
    for b, p in enumerate(pts):
        xyz[b, :, :lengths[b]] = p.t()
    idx = torch.ops.ri.furthest_point_sample(xyz, torch.tensor(lengths, dtype=torch.int32), int(num_samples))
    safe = idx.clamp(min=0)
    points = _backend.gather_features_forward(xyz, safe).transpose(1, 2).contiguous()
    features = None
    if has_f:
        C = feats[0].shape[1]
        if any(f.dim() != 2 or f.shape != (n, C) for f, n in zip(feats, lengths)):
            raise RuntimeError("features must be [n_b, C] with one C for every cloud")
        fb = torch.zeros((B, C, N), dtype=torch.float32, device=dev)
        for b, f in enumerate(feats):
            fb[b, :, :lengths[b]] = torch.as_tensor(f, dtype=torch.float32, device=dev).t()
        features = _backend.gather_features_forward(fb, safe).transpose(1, 2).contiguous()
    return points, features, idx
