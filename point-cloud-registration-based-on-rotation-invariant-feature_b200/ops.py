"""torch custom ops (`torch.ops.ri.*`) over the C ABI of libri_b200.so.

This is the thin registration layer the north star asks for: every op checks its tensors the way the reference's
C++ wrappers do (CUDA / contiguous / dtype — utils.hpp:15-28 — raising RuntimeError), allocates the outputs with
torch (so they live in the caching allocator, as the reference's torch::zeros outputs do), and enqueues the
hand-written sm_100a kernels on torch's CURRENT stream through ctypes.  There is no other implementation behind
these names: no Triton, no eager fallback, no CPU path.
"""
import ctypes
import math
from typing import Optional

import torch

from . import _lib

_L = _lib.lib
_check = _lib.check


def _req(t, name, dtype):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor" % name)
    if not t.is_contiguous():
        raise RuntimeError("%s must be a contiguous tensor" % name)
    if t.dtype != dtype:
        raise RuntimeError("%s must be %s tensor" % (name, "a float" if dtype == torch.float32 else "an int"))


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _same_device(*ts):
    d = ts[0].device
    for t in ts[1:]:
        if t.device != d:
            raise RuntimeError("all tensors must be on the same device")
    return d


def _shape(t, name, *want):
    """Raise (before anything is enqueued) unless t has exactly the dimensions `want` (None = any size)."""
    if t.dim() != len(want) or any(w is not None and int(d) != int(w) for d, w in zip(t.shape, want)):
        raise RuntimeError("%s must have shape [%s], got %s" % (name, ", ".join("*" if w is None else str(w) for w in want),
                                                               list(t.shape)))


_WS = {}
_WS_MAX = 8        # scratch buffers kept alive: (device, stream) pairs come and go, the cache must not grow with them


def _workspace(device, nbytes):
    """Per-(device, stream) scratch buffer for the voxelizer (stream-ordered reuse is safe on one stream).  The cache holds
    the _WS_MAX most recently used buffers; an evicted buffer is freed by the caching allocator in stream order."""
    key = (device, _stream())
    buf = _WS.pop(key, None)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8, device=device)
    _WS[key] = buf                                   # re-inserted last: dicts keep insertion order
    while len(_WS) > _WS_MAX:
        _WS.pop(next(iter(_WS)))
    return buf


# ---------------------------------------------------------------------------------------------- KNN
def _check_knn_shapes(xyz1, xyz2, k):
    if xyz1.dim() != 3 or xyz2.dim() != 3:
        raise RuntimeError("xyz1 / xyz2 must be [B, c, n] / [B, c, m] tensors")
    if xyz1.shape[0] != xyz2.shape[0] or xyz1.shape[1] != xyz2.shape[1]:
        raise RuntimeError("xyz1 and xyz2 must agree in batch size and channel count")
    if k <= 0:
        raise RuntimeError("k must be positive")


GRID_KNN_MIN_REFS = 4096     # at and above this many reference points (c == 3, k <= 32) the hash-grid search is used


def _knn_dir(q, r, B, c, n, m, k, d, i, dev):
    """One direction of the k-NN: brute force for small clouds, uniform hash grid for scan-sized ones.  Both produce
    the same bits (csrc/knn_grid.cu); this is an algorithm choice by problem size, not a backend switch."""
    if c == 3 and k <= 32 and m >= GRID_KNN_MIN_REFS:
        nws = _L.ri_knn_grid_workspace_bytes(B, n, m)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_knn_grid_f32(q.data_ptr(), r.data_ptr(), B, n, m, k, d.data_ptr(), i.data_ptr(),
                                  ws.data_ptr(), nws, _stream()), "ri_knn_grid")
    else:
        _check(_L.ri_knn_f32(q.data_ptr(), r.data_ptr(), B, c, n, m, k, d.data_ptr(), i.data_ptr(), _stream()), "ri_knn")

@torch.library.custom_op("ri::knn", mutates_args=())
def knn(xyz1: torch.Tensor, xyz2: torch.Tensor, k: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    _req(xyz1, "xyz1", torch.float32); _req(xyz2, "xyz2", torch.float32)
    dev = _same_device(xyz1, xyz2)
    _check_knn_shapes(xyz1, xyz2, k)
    B, c, n = xyz1.shape
    m = xyz2.shape[2]
    with torch.cuda.device(dev):
        d1 = torch.empty((B, k, n), dtype=torch.float32, device=dev)
        d2 = torch.empty((B, k, m), dtype=torch.float32, device=dev)
        i1 = torch.empty((B, k, n), dtype=torch.int32, device=dev)
        i2 = torch.empty((B, k, m), dtype=torch.int32, device=dev)
        if c == 3 and k <= 32 and max(n, m) >= GRID_KNN_MIN_REFS:
            _knn_dir(xyz1, xyz2, B, c, n, m, k, d1, i1, dev)
            _knn_dir(xyz2, xyz1, B, c, m, n, k, d2, i2, dev)
        else:
            _check(_L.ri_knn_bilateral_f32(xyz1.data_ptr(), xyz2.data_ptr(), B, c, n, m, k,
                                           d1.data_ptr(), d2.data_ptr(), i1.data_ptr(), i2.data_ptr(), _stream()), "ri_knn")
    return d1, d2, i1, i2


@knn.register_fake
def _(xyz1, xyz2, k):
    B, c, n = xyz1.shape
    m = xyz2.shape[2]
    return (xyz1.new_empty((B, k, n)), xyz1.new_empty((B, k, m)),
            xyz1.new_empty((B, k, n), dtype=torch.int32), xyz1.new_empty((B, k, m), dtype=torch.int32))


@torch.library.custom_op("ri::knn_one", mutates_args=())
def knn_one(xyz1: torch.Tensor, xyz2: torch.Tensor, k: int) -> tuple[torch.Tensor, torch.Tensor]:
    """One direction only (queries xyz1 against references xyz2)."""
    _req(xyz1, "xyz1", torch.float32); _req(xyz2, "xyz2", torch.float32)
    dev = _same_device(xyz1, xyz2)
    _check_knn_shapes(xyz1, xyz2, k)
    B, c, n = xyz1.shape
    m = xyz2.shape[2]
    with torch.cuda.device(dev):
        d1 = torch.empty((B, k, n), dtype=torch.float32, device=dev)
        i1 = torch.empty((B, k, n), dtype=torch.int32, device=dev)
        _knn_dir(xyz1, xyz2, B, c, n, m, k, d1, i1, dev)
    return d1, i1


@torch.library.custom_op("ri::knn_brute", mutates_args=())
def knn_brute(xyz1: torch.Tensor, xyz2: torch.Tensor, k: int) -> tuple[torch.Tensor, torch.Tensor]:
    """One direction through the one-thread-per-query kernel regardless of size (csrc/knn.cu) — what the warp-per-query
    kernel (csrc/knn_warp.cu) must equal."""
    _req(xyz1, "xyz1", torch.float32); _req(xyz2, "xyz2", torch.float32)
    dev = _same_device(xyz1, xyz2)
    B, c, n = xyz1.shape
    m = xyz2.shape[2]
    _check_knn_shapes(xyz1, xyz2, k)
    with torch.cuda.device(dev):
        d1 = torch.empty((B, k, n), dtype=torch.float32, device=dev)
        i1 = torch.empty((B, k, n), dtype=torch.int32, device=dev)
        _check(_L.ri_knn_thread_f32(xyz1.data_ptr(), xyz2.data_ptr(), B, c, n, m, k, d1.data_ptr(), i1.data_ptr(), _stream()), "ri_knn")
    return d1, i1


@knn_brute.register_fake
def _(xyz1, xyz2, k):
    B, c, n = xyz1.shape
    return xyz1.new_empty((B, k, n)), xyz1.new_empty((B, k, n), dtype=torch.int32)


@torch.library.custom_op("ri::knn_grid", mutates_args=())
def knn_grid(xyz1: torch.Tensor, xyz2: torch.Tensor, k: int) -> tuple[torch.Tensor, torch.Tensor]:
    """One direction through the hash grid regardless of size (c == 3, k <= 32)."""
    _req(xyz1, "xyz1", torch.float32); _req(xyz2, "xyz2", torch.float32)
    dev = _same_device(xyz1, xyz2)
    B, c, n = xyz1.shape
    m = xyz2.shape[2]
    if c != 3 or xyz2.shape[1] != 3:
        raise RuntimeError("knn_grid needs 3-channel coordinates")
    with torch.cuda.device(dev):
        d1 = torch.empty((B, k, n), dtype=torch.float32, device=dev)
        i1 = torch.empty((B, k, n), dtype=torch.int32, device=dev)
        nws = _L.ri_knn_grid_workspace_bytes(B, n, m)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_knn_grid_f32(xyz1.data_ptr(), xyz2.data_ptr(), B, n, m, k, d1.data_ptr(), i1.data_ptr(),
                                  ws.data_ptr(), nws, _stream()), "ri_knn_grid")
    return d1, i1


@knn_grid.register_fake
def _(xyz1, xyz2, k):
    B, c, n = xyz1.shape
    return xyz1.new_empty((B, k, n)), xyz1.new_empty((B, k, n), dtype=torch.int32)


@knn_one.register_fake
def _(xyz1, xyz2, k):
    B, c, n = xyz1.shape
    return xyz1.new_empty((B, k, n)), xyz1.new_empty((B, k, n), dtype=torch.int32)


@torch.library.custom_op("ri::knn_backward", mutates_args=())
def knn_backward(xyz1: torch.Tensor, xyz2: torch.Tensor, graddist1: torch.Tensor, graddist2: torch.Tensor,
                 idx1: torch.Tensor, idx2: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    for t, nm in ((xyz1, "xyz1"), (xyz2, "xyz2"), (graddist1, "graddist1"), (graddist2, "graddist2")):
        _req(t, nm, torch.float32)
    _req(idx1, "idx1", torch.int32); _req(idx2, "idx2", torch.int32)
    dev = _same_device(xyz1, xyz2, graddist1, graddist2, idx1, idx2)
    B, c, n = xyz1.shape
    m = xyz2.shape[2]
    k = idx1.shape[1]
    with torch.cuda.device(dev):
        g1 = torch.empty_like(xyz1); g2 = torch.empty_like(xyz2)
        _check(_L.ri_knn_backward_f32(xyz1.data_ptr(), xyz2.data_ptr(), graddist1.data_ptr(), graddist2.data_ptr(),
                                      idx1.data_ptr(), idx2.data_ptr(), B, c, n, m, k, g1.data_ptr(), g2.data_ptr(),
                                      _stream()), "ri_knn_backward")
    return g1, g2


@knn_backward.register_fake
def _(xyz1, xyz2, graddist1, graddist2, idx1, idx2):
    return torch.empty_like(xyz1), torch.empty_like(xyz2)


# ---------------------------------------------------------------------------------------------- PPF
@torch.library.custom_op("ri::ppf", mutates_args=())
def ppf(coords: torch.Tensor, center: torch.Tensor, normals: torch.Tensor, center_normal: torch.Tensor) -> torch.Tensor:
    """Backend argument order of spherical_ppf_forward (points first, centres second)."""
    for t, nm in ((coords, "coords"), (center, "center"), (normals, "normals"), (center_normal, "center_normal")):
        _req(t, nm, torch.float32)
    dev = _same_device(coords, center, normals, center_normal)
    _shape(coords, "coords", None, 3, None)
    B, _, L = coords.shape
    for t, nm in ((center, "center"), (normals, "normals"), (center_normal, "center_normal")):
        _shape(t, nm, B, 3, L)
    with torch.cuda.device(dev):
        feat = torch.empty((B, 4, L), dtype=torch.float32, device=dev)
        _check(_L.ri_ppf_f32(coords.data_ptr(), center.data_ptr(), normals.data_ptr(), center_normal.data_ptr(),
                             B, L, feat.data_ptr(), _stream()), "ri_ppf")
    return feat


@ppf.register_fake
def _(coords, center, normals, center_normal):
    B, _, L = coords.shape
    return coords.new_empty((B, 4, L))


@torch.library.custom_op("ri::ppf_gather", mutates_args=())
def ppf_gather(xyz: torch.Tensor, normals: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    _req(xyz, "xyz", torch.float32); _req(normals, "normals", torch.float32); _req(idx, "idx", torch.int32)
    dev = _same_device(xyz, normals, idx)
    _shape(xyz, "xyz", None, 3, None)
    B, _, N = xyz.shape
    _shape(normals, "normals", B, 3, N); _shape(idx, "idx", B, None, N)
    k = idx.shape[1]
    with torch.cuda.device(dev):
        out = torch.empty((B, 4, k, N), dtype=torch.float32, device=dev)
        _check(_L.ri_ppf_gather_f32(xyz.data_ptr(), normals.data_ptr(), idx.data_ptr(), B, N, k, out.data_ptr(), _stream()),
               "ri_ppf_gather")
    return out


@ppf_gather.register_fake
def _(xyz, normals, idx):
    B, _, N = xyz.shape
    return xyz.new_empty((B, 4, idx.shape[1], N))


# --------------------------------------------------------------------------------------- voxelization
def _voxelize(fn, what, features, coords, r, coord_dtype):
    _req(features, "features", torch.float32); _req(coords, "coords", coord_dtype)
    dev = _same_device(features, coords)
    _shape(features, "features", None, None, None)
    B, C, N = features.shape
    _shape(coords, "coords", B, 3, N)
    if r <= 0:
        raise RuntimeError("resolution must be positive")
    s = r * r * r
    with torch.cuda.device(dev):
        out = torch.empty((B, C, s), dtype=torch.float32, device=dev)
        ind = torch.empty((B, N), dtype=torch.int32, device=dev)
        cnt = torch.empty((B, s), dtype=torch.int32, device=dev)
        nbytes = _L.ri_voxelize_workspace_bytes(B, C, N, r)
        ws = _workspace(dev, nbytes)
        _check(fn(features.data_ptr(), coords.data_ptr(), B, C, N, r, out.data_ptr(), ind.data_ptr(), cnt.data_ptr(),
                  ws.data_ptr(), ws.numel(), _stream()), what)
    return out, ind, cnt


@torch.library.custom_op("ri::sph_voxelize", mutates_args=())
def sph_voxelize(features: torch.Tensor, coords: torch.Tensor, r: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return _voxelize(_L.ri_sph_voxelize_f32, "ri_sph_voxelize", features, coords, r, torch.float32)


@torch.library.custom_op("ri::cube_voxelize", mutates_args=())
def cube_voxelize(features: torch.Tensor, coords: torch.Tensor, r: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return _voxelize(_L.ri_cube_voxelize_f32, "ri_cube_voxelize", features, coords, r, torch.int32)


def _voxelize_edge(fn, what, features, coords, r, coord_dtype):
    _req(features, "features", torch.float32); _req(coords, "coords", coord_dtype)
    dev = _same_device(features, coords)
    _shape(features, "features", None, None, None)
    B, C, N = features.shape
    _shape(coords, "coords", B, 3, N)
    if r <= 0:
        raise RuntimeError("resolution must be positive")
    s = r * r * r
    with torch.cuda.device(dev):
        out = torch.empty((B, C, s), dtype=torch.float32, device=dev)
        ind = torch.empty((B, N), dtype=torch.int32, device=dev)
        cnt = torch.empty((B, s), dtype=torch.int32, device=dev)
        edge = torch.empty((B, 2 * C, N), dtype=torch.float32, device=dev)
        ws = _workspace(dev, _L.ri_voxelize_workspace_bytes(B, C, N, r))
        _check(fn(features.data_ptr(), coords.data_ptr(), B, C, N, r, out.data_ptr(), ind.data_ptr(), cnt.data_ptr(),
                  edge.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), what)
    return out, ind, cnt, edge


@torch.library.custom_op("ri::sph_voxelize_edge", mutates_args=())
def sph_voxelize_edge(features: torch.Tensor, coords: torch.Tensor, r: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    return _voxelize_edge(_L.ri_sph_voxelize_edge_f32, "ri_sph_voxelize_edge", features, coords, r, torch.float32)


@torch.library.custom_op("ri::cube_voxelize_edge", mutates_args=())
def cube_voxelize_edge(features: torch.Tensor, coords: torch.Tensor, r: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    return _voxelize_edge(_L.ri_cube_voxelize_edge_f32, "ri_cube_voxelize_edge", features, coords, r, torch.int32)


def _vox_edge_fake(features, coords, r):
    B, C, N = features.shape
    s = r * r * r
    return (features.new_empty((B, C, s)), features.new_empty((B, N), dtype=torch.int32),
            features.new_empty((B, s), dtype=torch.int32), features.new_empty((B, 2 * C, N)))


sph_voxelize_edge.register_fake(_vox_edge_fake)
cube_voxelize_edge.register_fake(_vox_edge_fake)


def _vox_fake(features, coords, r):
    B, C, N = features.shape
    s = r * r * r
    return (features.new_empty((B, C, s)), features.new_empty((B, N), dtype=torch.int32),
            features.new_empty((B, s), dtype=torch.int32))


sph_voxelize.register_fake(_vox_fake)
cube_voxelize.register_fake(_vox_fake)


@torch.library.custom_op("ri::voxelize_backward", mutates_args=())
def voxelize_backward(grad_y: torch.Tensor, ind: torch.Tensor, cnt: torch.Tensor) -> torch.Tensor:
    _req(grad_y, "grad_y", torch.float32); _req(ind, "indices", torch.int32); _req(cnt, "cnt", torch.int32)
    dev = _same_device(grad_y, ind, cnt)
    B, C, s = grad_y.shape
    N = ind.shape[1]
    with torch.cuda.device(dev):
        gx = torch.empty((B, C, N), dtype=torch.float32, device=dev)
        _check(_L.ri_voxelize_backward_f32(grad_y.data_ptr(), ind.data_ptr(), cnt.data_ptr(), B, C, N, s,
                                           gx.data_ptr(), _stream()), "ri_voxelize_backward")
    return gx


@voxelize_backward.register_fake
def _(grad_y, ind, cnt):
    return grad_y.new_empty((grad_y.shape[0], grad_y.shape[1], ind.shape[1]))


# ------------------------------------------------------------------------------------- devoxelization
@torch.library.custom_op("ri::trilinear_devox", mutates_args=())
def trilinear_devox(coords: torch.Tensor, features: torch.Tensor, r: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    _req(features, "features", torch.float32); _req(coords, "coords", torch.float32)
    dev = _same_device(features, coords)
    B, C = features.shape[:2]
    _shape(coords, "coords", B, 3, None)
    N = coords.shape[2]
    if r <= 0 or features.numel() != B * C * r ** 3:
        raise RuntimeError("features must hold B*C*r^3 elements")
    with torch.cuda.device(dev):
        outs = torch.empty((B, C, N), dtype=torch.float32, device=dev)
        inds = torch.empty((B, 8, N), dtype=torch.int32, device=dev)
        wgts = torch.empty((B, 8, N), dtype=torch.float32, device=dev)
        _check(_L.ri_trilinear_devox_f32(coords.data_ptr(), features.data_ptr(), B, C, N, r,
                                         outs.data_ptr(), inds.data_ptr(), wgts.data_ptr(), _stream()), "ri_trilinear_devox")
    return outs, inds, wgts


@torch.library.custom_op("ri::sph_trilinear_devox", mutates_args=())
def sph_trilinear_devox(coords: torch.Tensor, features: torch.Tensor, g_inds: torch.Tensor, r: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    _req(features, "features", torch.float32); _req(coords, "coords", torch.float32); _req(g_inds, "g_inds", torch.int32)
    dev = _same_device(features, coords, g_inds)
    B, C = features.shape[:2]
    _shape(coords, "coords", B, 3, None)
    N = coords.shape[2]
    _shape(g_inds, "g_inds", B, N)
    if r <= 0 or features.numel() != B * C * r ** 3:
        raise RuntimeError("features must hold B*C*r^3 elements")
    if r < 4:
        raise RuntimeError("spherical devoxelization needs r >= 4: its corner indices reach r^2 + 7r + 4")
    with torch.cuda.device(dev):
        outs = torch.empty((B, C, N), dtype=torch.float32, device=dev)
        inds = torch.empty((B, 8, N), dtype=torch.int32, device=dev)
        wgts = torch.empty((B, 8, N), dtype=torch.float32, device=dev)
        _check(_L.ri_sph_trilinear_devox_f32(coords.data_ptr(), features.data_ptr(), g_inds.data_ptr(), B, C, N, r,
                                             outs.data_ptr(), inds.data_ptr(), wgts.data_ptr(), _stream()),
               "ri_sph_trilinear_devox")
    return outs, inds, wgts


def _devox_fake(coords, features, *rest):
    B, C = features.shape[:2]
    N = coords.shape[2]
    return (features.new_empty((B, C, N)), features.new_empty((B, 8, N), dtype=torch.int32), features.new_empty((B, 8, N)))


trilinear_devox.register_fake(_devox_fake)
sph_trilinear_devox.register_fake(_devox_fake)


@torch.library.custom_op("ri::devox_backward", mutates_args=())
def devox_backward(grad_y: torch.Tensor, inds: torch.Tensor, wgts: torch.Tensor, r: int, skip_undefined: bool) -> torch.Tensor:
    _req(grad_y, "grad_y", torch.float32); _req(inds, "indices", torch.int32); _req(wgts, "weights", torch.float32)
    dev = _same_device(grad_y, inds, wgts)
    B, C, N = grad_y.shape
    s = r ** 3
    with torch.cuda.device(dev):
        gx = torch.empty((B, C, s), dtype=torch.float32, device=dev)
        _check(_L.ri_devox_backward_f32(grad_y.data_ptr(), inds.data_ptr(), wgts.data_ptr(), B, C, N, s,
                                        int(skip_undefined), gx.data_ptr(), _stream()), "ri_devox_backward")
    return gx


@devox_backward.register_fake
def _(grad_y, inds, wgts, r, skip_undefined):
    return grad_y.new_empty((grad_y.shape[0], grad_y.shape[1], r ** 3))


# ------------------------------------------------------------------------------- DGCNN edge features
@torch.library.custom_op("ri::voxel_edge_gather", mutates_args=())
def voxel_edge_gather(avg: torch.Tensor, features: torch.Tensor, inds: torch.Tensor) -> torch.Tensor:
    _req(avg, "avg_voxel_features", torch.float32); _req(features, "features", torch.float32); _req(inds, "inds", torch.int32)
    dev = _same_device(avg, features, inds)
    B, C, N = features.shape
    s = avg.numel() // max(B * C, 1)
    with torch.cuda.device(dev):
        out = torch.empty((B, 2 * C, N), dtype=torch.float32, device=dev)
        _check(_L.ri_voxel_edge_gather_f32(avg.data_ptr(), features.data_ptr(), inds.data_ptr(), B, C, N, s,
                                           out.data_ptr(), _stream()), "ri_voxel_edge_gather")
    return out


@voxel_edge_gather.register_fake
def _(avg, features, inds):
    B, C, N = features.shape
    return features.new_empty((B, 2 * C, N))


@torch.library.custom_op("ri::knn_ppf", mutates_args=())
def knn_ppf(xyz: torch.Tensor, normals: torch.Tensor, k: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Self-query k-NN and the PPF of every (point, neighbour) pair: xyz, normals [B,3,N] -> dist [B,k,N], idx [B,k,N],
    ppf [B,4,k,N].  Up to 1024 points: the warp-per-query k-NN followed by the gather/PPF kernel (39 + 16 us at 32 x 1024,
    k = 20, against 127 us for the fused thread-per-query kernel); up to 2048 points and k <= 32: the fused kernel
    (ri_knn_ppf_f32); larger: the hash-grid k-NN + gather/PPF.  Same values on every path."""
    _req(xyz, "xyz", torch.float32); _req(normals, "normals", torch.float32)
    dev = _same_device(xyz, normals)
    B, c, N = xyz.shape
    if c != 3 or tuple(normals.shape) != (B, 3, N):
        raise RuntimeError("xyz and normals must both be [B,3,N]")
    with torch.cuda.device(dev):
        d = torch.empty((B, k, N), dtype=torch.float32, device=dev)
        i = torch.empty((B, k, N), dtype=torch.int32, device=dev)
        out = torch.empty((B, 4, k, N), dtype=torch.float32, device=dev)
        if 1024 < N <= 2048 and k <= 32:
            _check(_L.ri_knn_ppf_f32(xyz.data_ptr(), normals.data_ptr(), 3 * N, B, N, k, d.data_ptr(), i.data_ptr(),
                                     out.data_ptr(), _stream()), "ri_knn_ppf")
        else:
            _knn_dir(xyz, xyz, B, 3, N, N, k, d, i, dev)
            _check(_L.ri_ppf_gather_f32(xyz.data_ptr(), normals.data_ptr(), i.data_ptr(), B, N, k, out.data_ptr(), _stream()),
                   "ri_ppf_gather")
    return d, i, out


@knn_ppf.register_fake
def _(xyz, normals, k):
    B, c, N = xyz.shape
    return xyz.new_empty((B, k, N)), xyz.new_empty((B, k, N), dtype=torch.int32), xyz.new_empty((B, 4, k, N))


# ---------------------------------------------------------------------------------- ball query + grouping
@torch.library.custom_op("ri::ball_query", mutates_args=())
def ball_query(centers_coords: torch.Tensor, points_coords: torch.Tensor, radius: float, num_neighbors: int) -> torch.Tensor:
    _req(centers_coords, "centers_coords", torch.float32); _req(points_coords, "points_coords", torch.float32)
    dev = _same_device(centers_coords, points_coords)
    _shape(centers_coords, "centers_coords", None, 3, None)
    B, _, M = centers_coords.shape
    _shape(points_coords, "points_coords", B, 3, None)
    N = points_coords.shape[2]
    if num_neighbors <= 0:
        raise RuntimeError("num_neighbors must be positive")
    with torch.cuda.device(dev):
        out = torch.empty((B, M, num_neighbors), dtype=torch.int32, device=dev)
        _check(_L.ri_ball_query_f32(centers_coords.data_ptr(), points_coords.data_ptr(), B, N, M, float(radius),
                                    int(num_neighbors), out.data_ptr(), _stream()), "ri_ball_query")
    return out


@ball_query.register_fake
def _(centers_coords, points_coords, radius, num_neighbors):
    return centers_coords.new_empty((centers_coords.shape[0], centers_coords.shape[2], num_neighbors), dtype=torch.int32)


@torch.library.custom_op("ri::grouping", mutates_args=())
def grouping(features: torch.Tensor, indices: torch.Tensor) -> torch.Tensor:
    _req(features, "features", torch.float32); _req(indices, "indices", torch.int32)
    dev = _same_device(features, indices)
    _shape(features, "features", None, None, None)
    B, C, N = features.shape
    _shape(indices, "indices", B, None, None)
    _, M, U = indices.shape
    with torch.cuda.device(dev):
        out = torch.empty((B, C, M, U), dtype=torch.float32, device=dev)
        _check(_L.ri_grouping_f32(features.data_ptr(), indices.data_ptr(), B, C, N, M, U, out.data_ptr(), _stream()),
               "ri_grouping")
    return out


@grouping.register_fake
def _(features, indices):
    return features.new_empty((features.shape[0], features.shape[1], indices.shape[1], indices.shape[2]))


@torch.library.custom_op("ri::grouping_backward", mutates_args=())
def grouping_backward(grad_y: torch.Tensor, indices: torch.Tensor, n: int) -> torch.Tensor:
    _req(grad_y, "grad_y", torch.float32); _req(indices, "indices", torch.int32)
    dev = _same_device(grad_y, indices)
    _shape(grad_y, "grad_y", None, None, None, None)
    B, C, M, U = grad_y.shape
    _shape(indices, "indices", B, M, U)
    with torch.cuda.device(dev):
        gx = torch.empty((B, C, n), dtype=torch.float32, device=dev)
        _check(_L.ri_grouping_backward_f32(grad_y.data_ptr(), indices.data_ptr(), B, C, n, M, U, gx.data_ptr(), _stream()),
               "ri_grouping_backward")
    return gx


@grouping_backward.register_fake
def _(grad_y, indices, n):
    return grad_y.new_empty((grad_y.shape[0], grad_y.shape[1], n))


# ---------------------------------------------------------------------------------------------- matcher
@torch.library.custom_op("ri::mutual_nn", mutates_args=())
def mutual_nn(desc1: torch.Tensor, desc2: torch.Tensor, point_major: bool) -> tuple[
        torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """find_correspondence_one_pair (datasets/deepgmr_mn40.py:232-244) for P pairs.
    desc [P,C,n] (point_major False) or [P,n,C] (True) -> corr12 [P,n1], corr21 [P,n2], dist12 [P,n1],
    idx1 [P,n1], idx2 [P,n1] (mutual matches, -1 padded), count [P]."""
    _req(desc1, "desc1", torch.float32); _req(desc2, "desc2", torch.float32)
    dev = _same_device(desc1, desc2)
    if desc1.dim() != 3 or desc2.dim() != 3 or desc1.shape[0] != desc2.shape[0]:
        raise RuntimeError("desc1/desc2 must be [P,C,n] (or [P,n,C]) with the same number of pairs")
    P = desc1.shape[0]
    if point_major:
        n1, C = desc1.shape[1], desc1.shape[2]; n2, C2 = desc2.shape[1], desc2.shape[2]
    else:
        C, n1 = desc1.shape[1], desc1.shape[2]; C2, n2 = desc2.shape[1], desc2.shape[2]
    if C != C2:
        raise RuntimeError("desc1 and desc2 must have the same number of channels")
    i32 = torch.int32
    corr12 = torch.empty((P, n1), dtype=i32, device=dev); corr21 = torch.empty((P, n2), dtype=i32, device=dev)
    dist12 = torch.empty((P, n1), dtype=torch.float32, device=dev)
    idx1 = torch.empty((P, n1), dtype=i32, device=dev); idx2 = torch.empty((P, n1), dtype=i32, device=dev)
    count = torch.empty((P,), dtype=i32, device=dev)
    with torch.cuda.device(dev):
        nws = _L.ri_mutual_nn_workspace_bytes(P, C, n1, n2)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_mutual_nn_tf32x3(desc1.data_ptr(), desc2.data_ptr(), P, C, n1, n2, 1 if point_major else 0,
                                      corr12.data_ptr(), corr21.data_ptr(), dist12.data_ptr(), idx1.data_ptr(),
                                      idx2.data_ptr(), count.data_ptr(), ws.data_ptr(), nws, _stream()), "ri_mutual_nn")
    return corr12, corr21, dist12, idx1, idx2, count


@mutual_nn.register_fake
def _(desc1, desc2, point_major):
    P = desc1.shape[0]
    n1 = desc1.shape[1] if point_major else desc1.shape[2]
    n2 = desc2.shape[1] if point_major else desc2.shape[2]
    i = lambda *s: desc1.new_empty(s, dtype=torch.int32)
    return i(P, n1), i(P, n2), desc1.new_empty((P, n1)), i(P, n1), i(P, n1), i(P)


@torch.library.custom_op("ri::mutual_nn_indices", mutates_args=())
def mutual_nn_indices(desc1: torch.Tensor, desc2: torch.Tensor, point_major: bool) -> tuple[
        torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """The same matcher without the distance output — what the reference method returns: corr12 [P,n1], corr21 [P,n2], idx1, idx2
    [P,n1] (mutual matches, -1 padded), count [P].  dist12 = NULL lets the library skip the re-evaluation pass and, for
    channel-major descriptors, the re-tiled image altogether (csrc/matcher.cu, tensor-map path)."""
    _req(desc1, "desc1", torch.float32); _req(desc2, "desc2", torch.float32)
    dev = _same_device(desc1, desc2)
    if desc1.dim() != 3 or desc2.dim() != 3 or desc1.shape[0] != desc2.shape[0]:
        raise RuntimeError("desc1/desc2 must be [P,C,n] (or [P,n,C]) with the same number of pairs")
    P = desc1.shape[0]
    if point_major:
        n1, C = desc1.shape[1], desc1.shape[2]; n2, C2 = desc2.shape[1], desc2.shape[2]
    else:
        C, n1 = desc1.shape[1], desc1.shape[2]; C2, n2 = desc2.shape[1], desc2.shape[2]
    if C != C2:
        raise RuntimeError("desc1 and desc2 must have the same number of channels")
    i32 = torch.int32
    corr12 = torch.empty((P, n1), dtype=i32, device=dev); corr21 = torch.empty((P, n2), dtype=i32, device=dev)
    idx1 = torch.empty((P, n1), dtype=i32, device=dev); idx2 = torch.empty((P, n1), dtype=i32, device=dev)
    count = torch.empty((P,), dtype=i32, device=dev)
    with torch.cuda.device(dev):
        nws = _L.ri_mutual_nn_workspace_bytes(P, C, n1, n2)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_mutual_nn_tf32x3(desc1.data_ptr(), desc2.data_ptr(), P, C, n1, n2, 1 if point_major else 0,
                                      corr12.data_ptr(), corr21.data_ptr(), None, idx1.data_ptr(),
                                      idx2.data_ptr(), count.data_ptr(), ws.data_ptr(), nws, _stream()), "ri_mutual_nn")
    return corr12, corr21, idx1, idx2, count


@mutual_nn_indices.register_fake
def _(desc1, desc2, point_major):
    P = desc1.shape[0]
    n1 = desc1.shape[1] if point_major else desc1.shape[2]
    n2 = desc2.shape[1] if point_major else desc2.shape[2]
    i = lambda *s: desc1.new_empty(s, dtype=torch.int32)
    return i(P, n1), i(P, n2), i(P, n1), i(P, n1), i(P)


# ---------------------------------------------------------------------------------------------- grid subsampling (f2)
@torch.library.custom_op("ri::grid_subsample", mutates_args=())
def grid_subsample(points: torch.Tensor, features: torch.Tensor, labels: torch.Tensor, grid_size: float) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """points [N,3] f32, features [N,d] f32 (d may be 0), labels [N,l] i32 (l may be 0) -> (sub_points [N,3], sub_features
    [N,d], sub_labels [N,l], count [1] i32): the first count[0] rows are the cells in ascending cell index
    (csrc/gridsub.cu; reference grid_subsampling.cpp:4-106).  No host synchronisation."""
    _req(points, "points", torch.float32); _req(features, "features", torch.float32); _req(labels, "labels", torch.int32)
    dev = _same_device(points, features, labels)
    N = points.shape[0]
    fdim, ldim = features.shape[1], labels.shape[1]
    with torch.cuda.device(dev):
        op = torch.empty((N, 3), dtype=torch.float32, device=dev)
        of = torch.empty((N, fdim), dtype=torch.float32, device=dev)
        ol = torch.empty((N, ldim), dtype=torch.int32, device=dev)
        cnt = torch.empty((1,), dtype=torch.int32, device=dev)
        nws = _L.ri_grid_subsample_workspace_bytes(N)
        ws = torch.empty(max(nws, 256), dtype=torch.uint8, device=dev)
        _check(_L.ri_grid_subsample_f32(points.data_ptr(), features.data_ptr() if fdim else None,
                                        labels.data_ptr() if ldim else None, N, fdim, ldim, float(grid_size),
                                        op.data_ptr(), of.data_ptr() if fdim else None, ol.data_ptr() if ldim else None,
                                        cnt.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "ri_grid_subsample")
    return op, of, ol, cnt


@grid_subsample.register_fake
def _(points, features, labels, grid_size):
    N = points.shape[0]
    return (points.new_empty((N, 3)), features.new_empty((N, features.shape[1])),
            labels.new_empty((N, labels.shape[1])), labels.new_empty((1,)))


# ---------------------------------------------------------------------------------------------- pose + metrics (f3)
@torch.library.custom_op("ri::pose_from_matches", mutates_args=())
def pose_from_matches(src: torch.Tensor, tgt: torch.Tensor, idx1: torch.Tensor, idx2: torch.Tensor, count: torch.Tensor,
                      hyps: int, inlier_dist: float, edge_similarity: float, refine_iters: int, seed: int) -> tuple[torch.Tensor, torch.Tensor]:
    """src [P,n1,3], tgt [P,n2,3] f32; idx1/idx2 [P,ld], count [P] i32 (mutual matches) -> (T [P,4,4] f32 src->tgt,
    inliers [P] i32).  hyps == 0: least squares over all matches.  csrc/pose.cu."""
    _req(src, "src", torch.float32); _req(tgt, "tgt", torch.float32)
    _req(idx1, "idx1", torch.int32); _req(idx2, "idx2", torch.int32); _req(count, "count", torch.int32)
    dev = _same_device(src, tgt, idx1, idx2, count)
    _shape(src, "src", None, None, 3)
    P, n1, _ = src.shape
    _shape(tgt, "tgt", P, None, 3)
    _shape(idx1, "idx1", P, None)
    _shape(idx2, "idx2", P, idx1.shape[1])
    _shape(count, "count", P)
    if int(refine_iters) < 1:
        raise RuntimeError("refine_iters must be >= 1")
    if not float(inlier_dist) > 0.0:
        raise RuntimeError("inlier_dist must be > 0")
    n2 = tgt.shape[1]
    ld = idx1.shape[1]
    with torch.cuda.device(dev):
        T = torch.empty((P, 4, 4), dtype=torch.float32, device=dev)
        inl = torch.empty((P,), dtype=torch.int32, device=dev)
        best = torch.empty((max(P, 1),), dtype=torch.int64, device=dev)
        _check(_L.ri_pose_from_matches_f32(src.data_ptr(), tgt.data_ptr(), idx1.data_ptr(), idx2.data_ptr(), count.data_ptr(),
                                           P, n1, n2, ld, int(hyps), float(inlier_dist), float(edge_similarity),
                                           int(refine_iters), int(seed) & 0xFFFFFFFFFFFFFFFF, T.data_ptr(), inl.data_ptr(),
                                           best.data_ptr(), _stream()), "ri_pose_from_matches")
    return T, inl


@pose_from_matches.register_fake
def _(src, tgt, idx1, idx2, count, hyps, inlier_dist, edge_similarity, refine_iters, seed):
    P = src.shape[0]
    return src.new_empty((P, 4, 4)), count.new_empty((P,))


@torch.library.custom_op("ri::registration_metrics", mutates_args=())
def registration_metrics(gt: torch.Tensor, est: torch.Tensor, pts: torch.Tensor) -> torch.Tensor:
    """gt, est [P,4,4] f32, pts [P,n,3] f32 -> [P,3] f64 = (RRE degrees, RTE, RMSE), deepgmr_mn40.py:121-126,152-164."""
    _req(gt, "gt", torch.float32); _req(est, "est", torch.float32); _req(pts, "pts", torch.float32)
    dev = _same_device(gt, est, pts)
    P, n, _ = pts.shape
    with torch.cuda.device(dev):
        out = torch.empty((P, 3), dtype=torch.float64, device=dev)
        _check(_L.ri_registration_metrics_f32(gt.data_ptr(), est.data_ptr(), pts.data_ptr(), P, n, out.data_ptr(), _stream()),
               "ri_registration_metrics")
    return out


@registration_metrics.register_fake
def _(gt, est, pts):
    return gt.new_empty((gt.shape[0], 3), dtype=torch.float64)


# ---------------------------------------------------------------------------------------------- LRF change_coords (f4)
@torch.library.custom_op("ri::lrf_change_coords", mutates_args=())
def lrf_change_coords(coords: torch.Tensor, mean: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """coords [B,3,N] or [B,6,N] f32, mean [B,3] f32 (coords[:, :3].mean(2)) -> (new_coords [B,3,N], bases [B,3,3], ok [B] i32).
    csrc/lrf.cu; reference PVCNN/models/pvcnn_classify.py:153-184."""
    _req(coords, "coords", torch.float32); _req(mean, "mean", torch.float32)
    dev = _same_device(coords, mean)
    B, cs, N = coords.shape
    if cs not in (3, 6):
        raise RuntimeError("coords must be [B,3,N] or [B,6,N]")
    with torch.cuda.device(dev):
        out = torch.empty((B, 3, N), dtype=torch.float32, device=dev)
        bases = torch.empty((B, 3, 3), dtype=torch.float32, device=dev)
        ok = torch.empty((B,), dtype=torch.int32, device=dev)
        _check(_L.ri_lrf_change_coords_f32(coords.data_ptr(), cs, mean.data_ptr(), B, N, 1, out.data_ptr(), bases.data_ptr(),
                                           ok.data_ptr(), _stream()), "ri_lrf_change_coords")
    return out, bases, ok


@lrf_change_coords.register_fake
def _(coords, mean):
    B, _, N = coords.shape
    return coords.new_empty((B, 3, N)), coords.new_empty((B, 3, 3)), coords.new_empty((B,), dtype=torch.int32)


# ---------------------------------------------------------------------------------------------- local PPF (f1, fused)
@torch.library.custom_op("ri::local_ppf", mutates_args=())
def local_ppf(points_coords: torch.Tensor, points_normals: torch.Tensor, centers_coords: torch.Tensor,
              centers_normals: torch.Tensor, neighbors: torch.Tensor) -> torch.Tensor:
    """points_* [B,3,N], centers_* [B,3,M] f32, neighbors [B,M,U] i32 -> [B,4,U,M] (pvcnn_classify.py:252-270)."""
    for t, n in ((points_coords, "points_coords"), (points_normals, "points_normals"), (centers_coords, "centers_coords"),
                 (centers_normals, "centers_normals")):
        _req(t, n, torch.float32)
    _req(neighbors, "neighbors", torch.int32)
    dev = _same_device(points_coords, points_normals, centers_coords, centers_normals, neighbors)
    _shape(points_coords, "points_coords", None, 3, None)
    B, _, N = points_coords.shape
    _shape(points_normals, "points_normals", B, 3, N); _shape(centers_coords, "centers_coords", B, 3, None)
    M = centers_coords.shape[2]
    _shape(centers_normals, "centers_normals", B, 3, M); _shape(neighbors, "neighbors", B, M, None)
    U = neighbors.shape[2]
    with torch.cuda.device(dev):
        out = torch.empty((B, 4, U, M), dtype=torch.float32, device=dev)
        _check(_L.ri_local_ppf_f32(points_coords.data_ptr(), points_normals.data_ptr(), centers_coords.data_ptr(),
                                   centers_normals.data_ptr(), neighbors.data_ptr(), B, N, M, U, out.data_ptr(), _stream()),
               "ri_local_ppf")
    return out


@local_ppf.register_fake
def _(points_coords, points_normals, centers_coords, centers_normals, neighbors):
    return points_coords.new_empty((points_coords.shape[0], 4, neighbors.shape[2], centers_coords.shape[2]))


@torch.library.custom_op("ri::local_ppf_mlp_max", mutates_args=())
def local_ppf_mlp_max(points_coords: torch.Tensor, points_normals: torch.Tensor, centers_coords: torch.Tensor,
                      centers_normals: torch.Tensor, neighbors: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor,
                      w2: torch.Tensor, b2: torch.Tensor) -> torch.Tensor:
    """The local-feature branch fused (pvcnn_classify.py:252-271): points_* [B,3,N], centers_* [B,3,M], neighbors [B,M,128] i32,
    BatchNorm-folded weights w1 [32,4], b1 [32], w2 [64,32], b2 [64] -> [B,64,M] = max over the neighbours of the two-layer MLP
    on the local point-pair features."""
    for t, n in ((points_coords, "points_coords"), (points_normals, "points_normals"), (centers_coords, "centers_coords"),
                 (centers_normals, "centers_normals"), (w1, "w1"), (b1, "b1"), (w2, "w2"), (b2, "b2")):
        _req(t, n, torch.float32)
    _req(neighbors, "neighbors", torch.int32)
    dev = _same_device(points_coords, points_normals, centers_coords, centers_normals, neighbors, w1, b1, w2, b2)
    _shape(points_coords, "points_coords", None, 3, None)
    B, _, N = points_coords.shape
    _shape(points_normals, "points_normals", B, 3, N); _shape(centers_coords, "centers_coords", B, 3, None)
    M = centers_coords.shape[2]
    _shape(centers_normals, "centers_normals", B, 3, M); _shape(neighbors, "neighbors", B, M, None)
    U = neighbors.shape[2]
    _shape(w1, "w1", None, 4); C1 = w1.shape[0]
    _shape(b1, "b1", C1); _shape(w2, "w2", None, C1); C2 = w2.shape[0]; _shape(b2, "b2", C2)
    with torch.cuda.device(dev):
        out = torch.empty((B, C2, M), dtype=torch.float32, device=dev)
        _check(_L.ri_local_ppf_mlp_max_f32(points_coords.data_ptr(), points_normals.data_ptr(), centers_coords.data_ptr(),
                                           centers_normals.data_ptr(), neighbors.data_ptr(), B, N, M, U,
                                           w1.data_ptr(), b1.data_ptr(), C1, w2.data_ptr(), b2.data_ptr(), C2,
                                           out.data_ptr(), _stream()), "ri_local_ppf_mlp_max")
    return out


@local_ppf_mlp_max.register_fake
def _(points_coords, points_normals, centers_coords, centers_normals, neighbors, w1, b1, w2, b2):
    return points_coords.new_empty((points_coords.shape[0], w2.shape[0], centers_coords.shape[2]))


# ---------------------------------------------------------------------------------------------- ICP refinement (f5)
@torch.library.custom_op("ri::icp", mutates_args=())
def icp(src: torch.Tensor, tgt: torch.Tensor, tgt_normals: Optional[torch.Tensor], init: torch.Tensor, r: float,
        point_to_plane: bool, max_iter: int, rel_fitness: float, rel_rmse: float, want_corr: bool) -> tuple[
        torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """src [P,n1,3], tgt [P,n2,3], tgt_normals [P,n2,3] or None, init [P,4,4] f32 -> (T [P,4,4] f32, fitness [P] f64,
    inlier_rmse [P] f64, iterations [P] i32, corr [P,n1] i32 (target index or -1 under T; [P,0] unless want_corr)).
    Open3D's registration_icp per pair, all pairs in one call (csrc/icp.cu); max_iter == 0 evaluates init."""
    _req(src, "src", torch.float32); _req(tgt, "tgt", torch.float32); _req(init, "init", torch.float32)
    ts = (src, tgt, init)
    if tgt_normals is not None:
        _req(tgt_normals, "tgt_normals", torch.float32)
        ts = ts + (tgt_normals,)
    dev = _same_device(*ts)
    _shape(src, "src", None, None, 3)
    P, n1, _ = src.shape
    _shape(tgt, "tgt", P, None, 3)
    n2 = tgt.shape[1]
    _shape(init, "init", P, 4, 4)
    if tgt_normals is not None:
        _shape(tgt_normals, "tgt_normals", P, n2, 3)
    elif point_to_plane:
        raise RuntimeError("point-to-plane ICP needs tgt_normals")
    with torch.cuda.device(dev):
        T = torch.empty((P, 4, 4), dtype=torch.float32, device=dev)
        fit = torch.empty((P,), dtype=torch.float64, device=dev)
        rmse = torch.empty((P,), dtype=torch.float64, device=dev)
        iters = torch.empty((P,), dtype=torch.int32, device=dev)
        corr = torch.empty((P, n1 if want_corr else 0), dtype=torch.int32, device=dev)
        nws = _L.ri_icp_workspace_bytes(P, n1, n2)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_icp_f32(src.data_ptr(), tgt.data_ptr(), tgt_normals.data_ptr() if tgt_normals is not None else None,
                             init.data_ptr(), P, n1, n2, float(r), int(point_to_plane), int(max_iter), float(rel_fitness),
                             float(rel_rmse), T.data_ptr(), fit.data_ptr(), rmse.data_ptr(), iters.data_ptr(),
                             corr.data_ptr() if want_corr else None, ws.data_ptr(), nws, _stream()), "ri_icp")
    return T, fit, rmse, iters, corr


@icp.register_fake
def _(src, tgt, tgt_normals, init, r, point_to_plane, max_iter, rel_fitness, rel_rmse, want_corr):
    P, n1 = src.shape[0], src.shape[1]
    return (src.new_empty((P, 4, 4)), src.new_empty((P,), dtype=torch.float64), src.new_empty((P,), dtype=torch.float64),
            src.new_empty((P,), dtype=torch.int32), src.new_empty((P, n1 if want_corr else 0), dtype=torch.int32))


# ---------------------------------------------------------------------------------------------- Generalized ICP (f9)
def check_generalized_icp(src, tgt, src_normals, tgt_normals, init, r, epsilon, max_iter):
    """Raise RuntimeError unless the arguments of generalized_icp are valid; a normals argument may be None here (the
    Python wrapper estimates it after this check, so a bad call launches nothing)."""
    ts = [(src, "src"), (tgt, "tgt"), (init, "init")]
    ts += [(t, nm) for t, nm in ((src_normals, "src_normals"), (tgt_normals, "tgt_normals")) if t is not None]
    for t, nm in ts:
        _req(t, nm, torch.float32)
    _same_device(*(t for t, _ in ts))
    _shape(src, "src", None, None, 3)
    P, n1, _ = src.shape
    _shape(tgt, "tgt", P, None, 3)
    _shape(init, "init", P, 4, 4)
    if src_normals is not None:
        _shape(src_normals, "src_normals", P, n1, 3)
    if tgt_normals is not None:
        _shape(tgt_normals, "tgt_normals", P, tgt.shape[1], 3)
    if n1 < 1 or tgt.shape[1] < 1:
        raise RuntimeError("src and tgt need at least one point per pair")
    if not float(r) > 0.0:
        raise RuntimeError("max_correspondence_distance must be > 0")
    if not (math.isfinite(float(epsilon)) and float(epsilon) > 0.0):
        raise RuntimeError("epsilon must be finite and > 0")
    if int(max_iter) < 0:
        raise RuntimeError("max_iter must be >= 0")


@torch.library.custom_op("ri::generalized_icp", mutates_args=())
def generalized_icp(src: torch.Tensor, tgt: torch.Tensor, src_normals: torch.Tensor, tgt_normals: torch.Tensor,
                    init: torch.Tensor, r: float, epsilon: float, max_iter: int, rel_fitness: float, rel_rmse: float,
                    want_corr: bool) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """src [P,n1,3], tgt [P,n2,3], src_normals [P,n1,3], tgt_normals [P,n2,3], init [P,4,4] f32 -> (T [P,4,4] f32,
    fitness [P] f64, inlier_rmse [P] f64, iterations [P] i32, corr [P,n1] i32 ([P,0] unless want_corr)).
    Open3D's registration_generalized_icp per pair, all pairs in one call (csrc/icp.cu); max_iter == 0 evaluates init."""
    check_generalized_icp(src, tgt, src_normals, tgt_normals, init, r, epsilon, max_iter)
    P, n1, _ = src.shape
    n2 = tgt.shape[1]
    dev = src.device
    with torch.cuda.device(dev):
        T = torch.empty((P, 4, 4), dtype=torch.float32, device=dev)
        fit = torch.empty((P,), dtype=torch.float64, device=dev)
        rmse = torch.empty((P,), dtype=torch.float64, device=dev)
        iters = torch.empty((P,), dtype=torch.int32, device=dev)
        corr = torch.empty((P, n1 if want_corr else 0), dtype=torch.int32, device=dev)
        nws = _L.ri_icp_workspace_bytes(P, n1, n2)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_generalized_icp_f32(src.data_ptr(), tgt.data_ptr(), src_normals.data_ptr(), tgt_normals.data_ptr(),
                                         init.data_ptr(), P, n1, n2, float(r), float(epsilon), int(max_iter),
                                         float(rel_fitness), float(rel_rmse), T.data_ptr(), fit.data_ptr(),
                                         rmse.data_ptr(), iters.data_ptr(), corr.data_ptr() if want_corr else None,
                                         ws.data_ptr(), nws, _stream()), "ri_generalized_icp")
    return T, fit, rmse, iters, corr


@generalized_icp.register_fake
def _(src, tgt, src_normals, tgt_normals, init, r, epsilon, max_iter, rel_fitness, rel_rmse, want_corr):
    P, n1 = src.shape[0], src.shape[1]
    return (src.new_empty((P, 4, 4)), src.new_empty((P,), dtype=torch.float64), src.new_empty((P,), dtype=torch.float64),
            src.new_empty((P,), dtype=torch.int32), src.new_empty((P, n1 if want_corr else 0), dtype=torch.int32))


# ---------------------------------------------------------------------------------------------- robust kernels (f11)
ROBUST_LOSSES = ('l2', 'l1', 'huber', 'cauchy', 'gm', 'tukey')      # position = RI_LOSS_* of include/ri_b200.h


def check_robust_icp(src, tgt, src_normals, tgt_normals, init, r, generalized, epsilon, loss, k, max_iter):
    """Raise RuntimeError unless the arguments of robust_icp are valid; a normals argument may be None here (the Python
    wrapper estimates generalized ICP's after this check, so a bad call launches nothing).  Point-to-plane reads neither
    src_normals nor epsilon."""
    check_generalized_icp(src, tgt, src_normals if generalized else None, tgt_normals, init, r,
                          epsilon if generalized else 1.0, max_iter)
    if not 0 <= int(loss) < len(ROBUST_LOSSES):
        raise RuntimeError("loss must be in [0, %d), got %r" % (len(ROBUST_LOSSES), loss))
    if int(loss) >= 2 and not (math.isfinite(float(k)) and float(k) > 0.0):
        raise RuntimeError("the %s kernel's parameter k must be finite and > 0, got %r" % (ROBUST_LOSSES[int(loss)], k))


@torch.library.custom_op("ri::robust_icp", mutates_args=())
def robust_icp(src: torch.Tensor, tgt: torch.Tensor, src_normals: Optional[torch.Tensor], tgt_normals: torch.Tensor,
               init: torch.Tensor, r: float, generalized: bool, epsilon: float, loss: int, k: float, max_iter: int,
               rel_fitness: float, rel_rmse: float, want_corr: bool) -> tuple[
               torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Point-to-plane (generalized=False: tgt_normals [P,n2,3]) or generalized ICP (src_normals [P,n1,3] too) with a robust
    kernel: loss = ROBUST_LOSSES.index(name), k its parameter.  Other arguments and the outputs as icp / generalized_icp.
    Open3D's TransformationEstimationPointToPlane(loss) / ForGeneralizedICP(epsilon, loss) per pair (csrc/icp.cu)."""
    check_robust_icp(src, tgt, src_normals, tgt_normals, init, r, generalized, epsilon, loss, k, max_iter)
    if tgt_normals is None or (generalized and src_normals is None):
        raise RuntimeError("robust_icp needs tgt_normals, and src_normals when generalized")
    P, n1, _ = src.shape
    n2 = tgt.shape[1]
    dev = src.device
    with torch.cuda.device(dev):
        T = torch.empty((P, 4, 4), dtype=torch.float32, device=dev)
        fit = torch.empty((P,), dtype=torch.float64, device=dev)
        rmse = torch.empty((P,), dtype=torch.float64, device=dev)
        iters = torch.empty((P,), dtype=torch.int32, device=dev)
        corr = torch.empty((P, n1 if want_corr else 0), dtype=torch.int32, device=dev)
        nws = _L.ri_icp_workspace_bytes(P, n1, n2)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_robust_icp_f32(src.data_ptr(), tgt.data_ptr(), src_normals.data_ptr() if generalized else None,
                                    tgt_normals.data_ptr(), init.data_ptr(), P, n1, n2, float(r), int(generalized),
                                    float(epsilon), int(loss), float(k), int(max_iter), float(rel_fitness),
                                    float(rel_rmse), T.data_ptr(), fit.data_ptr(), rmse.data_ptr(), iters.data_ptr(),
                                    corr.data_ptr() if want_corr else None, ws.data_ptr(), nws, _stream()),
               "ri_robust_icp")
    return T, fit, rmse, iters, corr


@robust_icp.register_fake
def _(src, tgt, src_normals, tgt_normals, init, r, generalized, epsilon, loss, k, max_iter, rel_fitness, rel_rmse,
      want_corr):
    P, n1 = src.shape[0], src.shape[1]
    return (src.new_empty((P, 4, 4)), src.new_empty((P,), dtype=torch.float64), src.new_empty((P,), dtype=torch.float64),
            src.new_empty((P,), dtype=torch.int32), src.new_empty((P, n1 if want_corr else 0), dtype=torch.int32))


# ---------------------------------------------------------------------------------------------- normal estimation (f6)
@torch.library.custom_op("ri::estimate_normals", mutates_args=())
def estimate_normals(xyz: torch.Tensor, radius: float, max_nn: int, camera: Optional[torch.Tensor],
                     prior: Optional[torch.Tensor]) -> tuple[torch.Tensor, torch.Tensor]:
    """xyz [B,3,N] f32, camera [B,3] or None, prior [B,3,N] or None -> (normals [B,3,N] f32, counts [B,N] i32).
    Open3D's estimate_normals with the hybrid (radius, max_nn) search, every cloud of the batch in one call
    (csrc/normals.cu); at most one of camera / prior orients the result."""
    _req(xyz, "xyz", torch.float32)
    ts = (xyz,)
    if camera is not None:
        _req(camera, "camera", torch.float32)
        ts = ts + (camera,)
    if prior is not None:
        _req(prior, "prior", torch.float32)
        ts = ts + (prior,)
    dev = _same_device(*ts)
    _shape(xyz, "xyz", None, 3, None)
    B, _, N = xyz.shape
    if camera is not None:
        _shape(camera, "camera", B, 3)
    if prior is not None:
        _shape(prior, "prior", B, 3, N)
    if camera is not None and prior is not None:
        raise RuntimeError("orient normals by a camera or by a prior, not both")
    with torch.cuda.device(dev):
        nrm = torch.empty((B, 3, N), dtype=torch.float32, device=dev)
        cnt = torch.empty((B, N), dtype=torch.int32, device=dev)
        nws = _L.ri_knn_grid_workspace_bytes(B, N, N)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_estimate_normals_f32(xyz.data_ptr(), B, N, float(radius), int(max_nn),
                                          camera.data_ptr() if camera is not None else None,
                                          prior.data_ptr() if prior is not None else None, nrm.data_ptr(), cnt.data_ptr(),
                                          ws.data_ptr(), nws, _stream()), "ri_estimate_normals")
    return nrm, cnt


@estimate_normals.register_fake
def _(xyz, radius, max_nn, camera, prior):
    B, _, N = xyz.shape
    return xyz.new_empty((B, 3, N)), xyz.new_empty((B, N), dtype=torch.int32)


# ---------------------------------------------------------------------------------------------- Fast Global Registration (f7)
@torch.library.custom_op("ri::fgr", mutates_args=())
def fgr(src: torch.Tensor, tgt: torch.Tensor, idx1: torch.Tensor, idx2: torch.Tensor, count: torch.Tensor,
        max_corr_dist: float, iterations: int, division_factor: float, use_absolute_scale: bool, decrease_mu: bool,
        tuple_test: bool, tuple_scale: float, max_tuples: int, seed: int, inlier_dist: float) -> tuple[
        torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """src [P,n1,3], tgt [P,n2,3] f32; idx1/idx2 [P,ld], count [P] i32 (mutual matches) -> (T [P,4,4] f32 src->tgt,
    inliers [P] i32, corr [P,3*max_tuples] i32 (the tuple list's match positions, -1 padded; [P,0] without the tuple test),
    ncorr [P] i32).  Open3D's FGR per pair, all pairs in one launch (csrc/fgr.cu)."""
    _req(src, "src", torch.float32); _req(tgt, "tgt", torch.float32)
    _req(idx1, "idx1", torch.int32); _req(idx2, "idx2", torch.int32); _req(count, "count", torch.int32)
    dev = _same_device(src, tgt, idx1, idx2, count)
    _shape(src, "src", None, None, 3)
    P, n1, _ = src.shape
    _shape(tgt, "tgt", P, None, 3)
    _shape(idx1, "idx1", P, None)
    _shape(idx2, "idx2", P, idx1.shape[1])
    _shape(count, "count", P)
    if not float(max_corr_dist) > 0.0:
        raise RuntimeError("maximum_correspondence_distance must be > 0")
    if int(iterations) < 0:
        raise RuntimeError("iteration_number must be >= 0")
    if not float(division_factor) > 1.0:
        raise RuntimeError("division_factor must be > 1")
    if not 0.0 < float(tuple_scale) <= 1.0:
        raise RuntimeError("tuple_scale must be in (0, 1]")
    if not 1 <= int(max_tuples) <= 0x7FFFFFFF // 3:
        raise RuntimeError("maximum_tuple_count must be in [1, %d]" % (0x7FFFFFFF // 3))
    if not float(inlier_dist) > 0.0:
        raise RuntimeError("inlier_dist must be > 0")
    n2 = tgt.shape[1]
    ld = idx1.shape[1]
    with torch.cuda.device(dev):
        T = torch.empty((P, 4, 4), dtype=torch.float32, device=dev)
        inl = torch.empty((P,), dtype=torch.int32, device=dev)
        corr = torch.empty((P, 3 * int(max_tuples) if tuple_test else 0), dtype=torch.int32, device=dev)
        ncorr = torch.empty((P,), dtype=torch.int32, device=dev)
        _check(_L.ri_fgr_f32(src.data_ptr(), tgt.data_ptr(), idx1.data_ptr(), idx2.data_ptr(), count.data_ptr(),
                             P, n1, n2, ld, float(max_corr_dist), int(iterations), float(division_factor),
                             int(use_absolute_scale), int(decrease_mu), int(tuple_test), float(tuple_scale), int(max_tuples),
                             int(seed) & 0xFFFFFFFFFFFFFFFF, float(inlier_dist), T.data_ptr(), inl.data_ptr(),
                             corr.data_ptr() if tuple_test else None, ncorr.data_ptr(), _stream()), "ri_fgr")
    return T, inl, corr, ncorr


@fgr.register_fake
def _(src, tgt, idx1, idx2, count, max_corr_dist, iterations, division_factor, use_absolute_scale, decrease_mu, tuple_test,
      tuple_scale, max_tuples, seed, inlier_dist):
    P = src.shape[0]
    return (src.new_empty((P, 4, 4)), count.new_empty((P,)), count.new_empty((P, 3 * max_tuples if tuple_test else 0)),
            count.new_empty((P,)))


# ---------------------------------------------------------------------------------------------- FPFH descriptors (f8)
@torch.library.custom_op("ri::compute_fpfh", mutates_args=())
def compute_fpfh(xyz: torch.Tensor, normals: torch.Tensor, radius: float, max_nn: int, with_spfh: bool,
                 with_counts: bool) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """xyz [B,3,N], normals [B,3,N] f32 -> (fpfh [B,33,N] f32, spfh [B,33,N] f32 ([0] unless with_spfh),
    counts [B,N] i32 ([0] unless with_counts)).  Open3D's compute_fpfh_feature with the hybrid (radius, max_nn) search,
    every cloud of the batch in one call (csrc/fpfh.cu)."""
    _req(xyz, "xyz", torch.float32); _req(normals, "normals", torch.float32)
    dev = _same_device(xyz, normals)
    _shape(xyz, "xyz", None, 3, None)
    B, _, N = xyz.shape
    _shape(normals, "normals", B, 3, N)
    if not float(radius) > 0.0:
        raise RuntimeError("radius must be > 0")
    if not 1 <= int(max_nn) <= 128:
        raise RuntimeError("max_nn must be in [1, 128]")
    if B > 65535:
        raise RuntimeError("at most 65535 clouds per call")
    with torch.cuda.device(dev):
        fpfh = torch.empty((B, 33, N), dtype=torch.float32, device=dev)
        spfh = torch.empty((B, 33, N) if with_spfh else (0,), dtype=torch.float32, device=dev)
        cnt = torch.empty((B, N) if with_counts else (0,), dtype=torch.int32, device=dev)
        nws = _L.ri_fpfh_workspace_bytes(B, N, int(max_nn))
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_compute_fpfh_f32(xyz.data_ptr(), normals.data_ptr(), B, N, float(radius), int(max_nn),
                                      fpfh.data_ptr(), spfh.data_ptr() if with_spfh else None,
                                      cnt.data_ptr() if with_counts else None, ws.data_ptr(), nws, _stream()),
               "ri_compute_fpfh")
    return fpfh, spfh, cnt


@compute_fpfh.register_fake
def _(xyz, normals, radius, max_nn, with_spfh, with_counts):
    B, _, N = xyz.shape
    return (xyz.new_empty((B, 33, N)), xyz.new_empty((B, 33, N) if with_spfh else (0,)),
            xyz.new_empty((B, N) if with_counts else (0,), dtype=torch.int32))


# ---------------------------------------------------------------------------------------------- TEASER++ (f10)
TEASER_MAX_LD = 1 << 15


@torch.library.custom_op("ri::teaser", mutates_args=())
def teaser(src: torch.Tensor, tgt: torch.Tensor, idx1: torch.Tensor, idx2: torch.Tensor, count: torch.Tensor,
           noise_bound: float, cbar2: float, gnc_factor: float, max_iterations: int, cost_threshold: float,
           max_clique_nodes: int, inlier_dist: float) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor,
                                                              torch.Tensor]:
    """src [P,n1,3], tgt [P,n2,3] f32; idx1/idx2 [P,ld], count [P] i32 (mutual matches) -> (T [P,4,4] f32 src->tgt,
    inliers [P] i32, clique [P,ld] i32 (ascending match positions, -1 padded), clique_size [P] i32, exact [P] i32).
    TEASER++ with a known scale per pair, all pairs in one call (csrc/teaser.cu)."""
    _req(src, "src", torch.float32); _req(tgt, "tgt", torch.float32)
    _req(idx1, "idx1", torch.int32); _req(idx2, "idx2", torch.int32); _req(count, "count", torch.int32)
    dev = _same_device(src, tgt, idx1, idx2, count)
    _shape(src, "src", None, None, 3)
    P, n1, _ = src.shape
    _shape(tgt, "tgt", P, None, 3)
    _shape(idx1, "idx1", P, None)
    _shape(idx2, "idx2", P, idx1.shape[1])
    _shape(count, "count", P)
    for name, v in (("noise_bound", noise_bound), ("cbar2", cbar2), ("inlier_dist", inlier_dist)):
        if not (math.isfinite(float(v)) and float(v) > 0.0):
            raise RuntimeError("%s must be finite and > 0" % name)
    if not float(gnc_factor) > 1.0:
        raise RuntimeError("rotation_gnc_factor must be > 1")
    if int(max_iterations) < 0:
        raise RuntimeError("rotation_max_iterations must be >= 0")
    if not 1 <= int(max_clique_nodes) < 1 << 63:
        raise RuntimeError("max_clique_nodes must be >= 1")
    n2 = tgt.shape[1]
    ld = idx1.shape[1]
    if ld > TEASER_MAX_LD or P > 65535:
        raise RuntimeError("ri_teaser: unsupported size (ld <= %d and P <= 65535)" % TEASER_MAX_LD)
    with torch.cuda.device(dev):
        T = torch.empty((P, 4, 4), dtype=torch.float32, device=dev)
        inl = torch.empty((P,), dtype=torch.int32, device=dev)
        clique = torch.empty((P, ld), dtype=torch.int32, device=dev)
        size = torch.empty((P,), dtype=torch.int32, device=dev)
        exact = torch.empty((P,), dtype=torch.int32, device=dev)
        if P == 0 or ld == 0 or n1 == 0 or n2 == 0:
            T.copy_(torch.eye(4, device=dev).expand(P, 4, 4)); inl.zero_(); size.zero_(); exact.fill_(1)
            return T, inl, clique, size, exact
        nws = _L.ri_teaser_workspace_bytes(P, ld)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _check(_L.ri_teaser_f32(src.data_ptr(), tgt.data_ptr(), idx1.data_ptr(), idx2.data_ptr(), count.data_ptr(),
                                P, n1, n2, ld, float(noise_bound), float(cbar2), float(gnc_factor), int(max_iterations),
                                float(cost_threshold), int(max_clique_nodes), float(inlier_dist), T.data_ptr(),
                                inl.data_ptr(), clique.data_ptr(), size.data_ptr(), exact.data_ptr(), ws.data_ptr(), nws,
                                _stream()), "ri_teaser")
    return T, inl, clique, size, exact


@teaser.register_fake
def _(src, tgt, idx1, idx2, count, noise_bound, cbar2, gnc_factor, max_iterations, cost_threshold, max_clique_nodes,
      inlier_dist):
    P, ld = idx1.shape
    return (src.new_empty((P, 4, 4)), count.new_empty((P,)), count.new_empty((P, ld)), count.new_empty((P,)),
            count.new_empty((P,)))


# ---------------------------------------------------------------------------------------------- farthest point sampling (f12)
def check_furthest_point_sample(xyz, lengths, m):
    """Every check of ri::furthest_point_sample, on the host and before anything is enqueued."""
    _req(xyz, "xyz", torch.float32)
    _shape(xyz, "xyz", None, 3, None)
    B, _, N = xyz.shape
    if int(m) < 1:
        raise RuntimeError("the number of samples must be >= 1")
    if N > _lib.FPS_MAX_POINTS:
        raise RuntimeError("farthest point sampling takes at most %d points per cloud, got N = %d" % (_lib.FPS_MAX_POINTS, N))
    if lengths is not None:
        if lengths.device.type != "cpu":
            raise RuntimeError("lengths must be a host (CPU) tensor: its values are checked before the launch")
        if lengths.dtype != torch.int32:
            raise RuntimeError("lengths must be an int32 tensor")
        _shape(lengths, "lengths", B)
        if B and (int(lengths.min()) < 0 or int(lengths.max()) > N):
            raise RuntimeError("lengths must lie in [0, N] = [0, %d]" % N)


@torch.library.custom_op("ri::furthest_point_sample", mutates_args=())
def furthest_point_sample(xyz: torch.Tensor, lengths: Optional[torch.Tensor], m: int) -> torch.Tensor:
    """xyz [B,3,N] f32 (CUDA), lengths [B] i32 on the host or None (every cloud has N points), m >= 1 -> idx [B,m] i32.
    Farthest point sampling from index 0 with fp64 distances, the lowest index on ties (csrc/fps.cu, include/ri_b200.h)."""
    check_furthest_point_sample(xyz, lengths, m)
    B, _, N = xyz.shape
    dev = xyz.device
    with torch.cuda.device(dev):
        lens = lengths.contiguous().to(dev, non_blocking=True) if lengths is not None else None
        idx = torch.empty((B, int(m)), dtype=torch.int32, device=dev)
        _check(_L.ri_furthest_point_sample_f32(xyz.data_ptr(), lens.data_ptr() if lens is not None else None, B, N, int(m),
                                               idx.data_ptr(), _stream()), "ri_furthest_point_sample")
    return idx


@furthest_point_sample.register_fake
def _(xyz, lengths, m):
    return xyz.new_empty((xyz.shape[0], m), dtype=torch.int32)


# ---------------------------------------------------------------------------------------------- ISS keypoints (f13)
def check_iss_keypoints(xyz, salient_radius, non_max_radius, gamma_21, gamma_32, min_neighbors):
    """Every check of ri::iss_keypoints, on the host and before anything is enqueued."""
    _req(xyz, "xyz", torch.float32)
    _shape(xyz, "xyz", None, 3, None)
    B, _, N = xyz.shape
    for name, v in (("salient_radius", salient_radius), ("non_max_radius", non_max_radius)):
        if not (math.isfinite(float(v)) and float(v) >= 0.0):
            raise RuntimeError("%s must be finite and >= 0 (0 = from the cloud's resolution)" % name)
    for name, v in (("gamma_21", gamma_21), ("gamma_32", gamma_32)):
        if not float(v) > 0.0:
            raise RuntimeError("%s must be > 0" % name)
    if int(min_neighbors) < 1:
        raise RuntimeError("min_neighbors must be >= 1")
    if B > 65535 or B * N > 0x7FFFFFFF:
        raise RuntimeError("ri_iss_keypoints: unsupported size (B <= 65535 and B * N <= 2^31 - 1)")


@torch.library.custom_op("ri::iss_keypoints", mutates_args=())
def iss_keypoints(xyz: torch.Tensor, salient_radius: float, non_max_radius: float, gamma_21: float, gamma_32: float,
                  min_neighbors: int, want_saliency: bool) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """xyz [B,3,N] f32 (CUDA) -> (idx [B,N] i32 (keypoints ascending, -1 after count[b]), count [B] i32,
    saliency [B,N] f64 ([0] unless want_saliency), radii [B,2] f32 (salient, non-max) as used).  Open3D's
    compute_iss_keypoints, every cloud of the batch in one call (csrc/iss.cu); a radius of 0 takes both radii from the
    cloud's resolution."""
    check_iss_keypoints(xyz, salient_radius, non_max_radius, gamma_21, gamma_32, min_neighbors)
    B, _, N = xyz.shape
    dev = xyz.device
    with torch.cuda.device(dev):
        idx = torch.empty((B, N), dtype=torch.int32, device=dev)
        count = torch.empty((B,), dtype=torch.int32, device=dev)
        sal = torch.empty((B, N) if want_saliency else (0,), dtype=torch.float64, device=dev)
        radii = torch.empty((B, 2), dtype=torch.float32, device=dev)
        if B == 0:
            return idx, count, sal, radii
        nws = _L.ri_iss_workspace_bytes(B, N)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        gamma = (ctypes.c_double * 2)(float(gamma_21), float(gamma_32))
        _check(_L.ri_iss_keypoints_f32(xyz.data_ptr(), B, N, float(salient_radius), float(non_max_radius), gamma,
                                       int(min_neighbors), idx.data_ptr(), count.data_ptr(),
                                       sal.data_ptr() if want_saliency else None, radii.data_ptr(), ws.data_ptr(), nws,
                                       _stream()), "ri_iss_keypoints")
    return idx, count, sal, radii


@iss_keypoints.register_fake
def _(xyz, salient_radius, non_max_radius, gamma_21, gamma_32, min_neighbors, want_saliency):
    B, _, N = xyz.shape
    return (xyz.new_empty((B, N), dtype=torch.int32), xyz.new_empty((B,), dtype=torch.int32),
            xyz.new_empty((B, N) if want_saliency else (0,), dtype=torch.float64), xyz.new_empty((B, 2)))
