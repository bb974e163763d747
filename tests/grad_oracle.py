"""Restatements of the front end's backward pass in plain torch — TEST INFRASTRUCTURE ONLY.

Every function computes in the dtype of its inputs and on their device; called with float64 tensors it is the fp64
oracle the gradient tests hold the CUDA kernels (csrc/grad.cu, csrc/ballquery.cu) and the autograd Functions
(functional/*.py) to.  Two kinds are given for each op:
  - the differentiable FORWARD, from the op's definition, so that fp64 autograd derives the gradient independently of any
    backward code of ours;
  - the BACKWARD written out (what the reference's gradient kernel computes), for the kernel-level tests.
Indices, counts and devoxelization corner weights are inputs, never recomputed here: they are not differentiable, and the
forward tests pin them bit for bit against the reference.  Nothing here needs a GPU."""
import torch

KNN_SKIP = 20000.0        # knn.cu:68 — a slot whose 2 * graddist reaches this contributes nothing


def _expand_index(idx, C):
    """[B, L] integer indices -> [B, C, L] int64, for gather / scatter_add along the last axis."""
    return idx.long().unsqueeze(1).expand(-1, C, -1)


# ---------------------------------------------------------------------------------------------------- k-NN
def _knn_dist_dir(q, ref, idx):
    B, c, n = q.shape
    k = idx.shape[1]
    nb = torch.gather(ref, 2, _expand_index(idx.reshape(B, k * n), c)).reshape(B, c, k, n)
    return ((q.unsqueeze(2) - nb) ** 2).sum(1)


def knn_dist(xyz1, xyz2, idx1, idx2):
    """k-NN squared distances through the given neighbour indices: dist1[b,q,i] = |x1_i - x2_idx1[b,q,i]|^2 and the mirror
    for dist2.  Sentinel slots (no q-th neighbour: index 0) are distances to reference point 0 here, which is what the
    gradient kernel differentiates; the forward stores 10000 in them instead."""
    return _knn_dist_dir(xyz1, xyz2, idx1), _knn_dist_dir(xyz2, xyz1, idx2)


def _knn_grad_dir(q, ref, gd, idx, gq, gref):
    B, c, n = q.shape
    k = idx.shape[1]
    g = 2 * gd
    # The rule tests the GRADIENT, not the distance (2x is exact in every float format, so fp64 decides as fp32 does).  A
    # sentinel slot (dist 10000, index 0) therefore still pushes 2g (x_i - ref_0) onto reference point 0 unless the
    # incoming gradient itself is >= 10000.
    g = torch.where(g >= KNN_SKIP, torch.zeros_like(g), g)
    ii = _expand_index(idx.reshape(B, k * n), c)
    nb = torch.gather(ref, 2, ii).reshape(B, c, k, n)
    t = g.unsqueeze(1) * (q.unsqueeze(2) - nb)                       # [B, c, k, n]
    gq += t.sum(2)
    gref.scatter_add_(2, ii, -t.reshape(B, c, k * n))


def knn_grad(xyz1, xyz2, graddist1, graddist2, idx1, idx2):
    """knn_backward_cuda (knn/knn.cu:52-78, both directions): grad1[i] += 2g (x1_i - x2_idx), grad2[idx] -= the same, and
    the mirror from (graddist2, idx2).  -> (gradxyz1 [B,c,n], gradxyz2 [B,c,m])."""
    g1, g2 = torch.zeros_like(xyz1), torch.zeros_like(xyz2)
    _knn_grad_dir(xyz1, xyz2, graddist1.to(xyz1.dtype), idx1, g1, g2)
    _knn_grad_dir(xyz2, xyz1, graddist2.to(xyz1.dtype), idx2, g2, g1)
    return g1, g2


# ------------------------------------------------------------------------------------------------ voxelize
def voxel_counts(ind, s):
    """Points per cell [B, s] (int64); ind == -1 joins no cell."""
    valid = ind >= 0
    return torch.zeros((ind.shape[0], s), dtype=torch.int64, device=ind.device).scatter_add_(
        1, ind.clamp(min=0).long(), valid.long())


def avg_voxelize(features, ind, s):
    """Voxel means [B,C,s]: out[b,c,v] = sum of features[b,c,i] over the points with ind[b,i] == v, divided by their
    count (vox.cu:49-73 == spherical_vox.cu:91-125).  ind == -1 (an undefined spherical point) joins no cell."""
    B, C, N = features.shape
    cnt = voxel_counts(ind, s).to(features.dtype)
    w = torch.where(ind >= 0, 1.0 / cnt.gather(1, ind.clamp(min=0).long()).clamp(min=1), torch.zeros_like(cnt[:, :1]))
    out = torch.zeros((B, C, s), dtype=features.dtype, device=features.device)
    return out.scatter_add(2, _expand_index(ind.clamp(min=0), C), features * w.unsqueeze(1))


def avg_voxelize_grad(grad_y, ind, cnt):
    """avg_voxelize_backward (vox.cu:87-111): grad_x[b,c,i] = 0 + grad_y[b,c,ind] * (1 / cnt[ind]); 0 where ind == -1."""
    B, C, s = grad_y.shape
    pos = ind.clamp(min=0).long()
    n = cnt.gather(1, pos).to(grad_y.dtype)
    g = 0.0 + torch.gather(grad_y, 2, _expand_index(pos, C)) * (1.0 / n.clamp(min=1)).unsqueeze(1)
    return torch.where(((ind >= 0) & (n > 0)).unsqueeze(1), g, torch.zeros_like(g))


# ---------------------------------------------------------------------------------------------- devoxelize
def devox(grid, inds, wgts):
    """Trilinear devoxelization through given corners: out[b,c,i] = sum_q wgts[b,q,i] * grid[b,c,inds[b,q,i]]
    (trilinear_devox.cu:22-106; the spherical form only differs in how it finds the corners).  grid [B,C,...] with s
    cells; undefined spherical points carry inds[b,0,i] = -1 and zero weights, so they read nothing."""
    B, C = grid.shape[:2]
    N = inds.shape[2]
    v = torch.gather(grid.reshape(B, C, -1), 2, _expand_index(inds.clamp(min=0).reshape(B, 8 * N), C))
    return (v.reshape(B, C, 8, N) * wgts.to(grid.dtype).unsqueeze(1)).sum(2)


def devox_grad(grad_y, inds, wgts, s, skip_undefined):
    """trilinear_devoxelize_backward (trilinear_devox.cu:120-163) / the spherical one (spherical_trilinear_devox.cu:150-194):
    grad_x[b,c,inds[b,q,i]] += wgts[b,q,i] * grad_y[b,c,i] over the 8 corners; with skip_undefined a point whose
    inds[b,0,i] == -1 adds nothing."""
    B, C, N = grad_y.shape
    w = wgts.to(grad_y.dtype)
    if skip_undefined:
        w = torch.where(inds[:, :1] == -1, torch.zeros_like(w), w)
    t = (grad_y.unsqueeze(2) * w.unsqueeze(1)).reshape(B, C, 8 * N)
    out = torch.zeros((B, C, s), dtype=grad_y.dtype, device=grad_y.device)
    return out.scatter_add_(2, _expand_index(inds.clamp(min=0).reshape(B, 8 * N), C), t)


# ------------------------------------------------------------------------------------------- edge features
def voxel_edge_features(avg, features, ind):
    """DGCNN voxel-neighbour edge features (pvconv.py:68-90): cat(features - avg[:, :, ind] (0 where ind == -1),
    features) [B,2C,N].  avg [B,C,r,r,r] or [B,C,s]."""
    B, C, N = features.shape
    centre = torch.gather(avg.reshape(B, C, -1), 2, _expand_index(ind.clamp(min=0), C))
    rel = torch.where((ind == -1).unsqueeze(1), torch.zeros_like(features), features - centre)
    return torch.cat((rel, features), 1)


# ----------------------------------------------------------------------------------------------- grouping
def grouping(features, indices):
    """grouping/grouping.cu:18-44: features [B,C,N], indices [B,M,U] -> features[b, c, indices[b,m,u]] [B,C,M,U]."""
    B, C, _ = features.shape
    _, M, U = indices.shape
    return torch.gather(features, 2, _expand_index(indices.reshape(B, M * U), C)).reshape(B, C, M, U)


def grouping_grad(grad_y, indices, n):
    """grouping/grouping.cu:58-84: grad_x[b,c,indices[b,m,u]] += grad_y[b,c,m,u] -> [B,C,n]."""
    B, C, M, U = grad_y.shape
    out = torch.zeros((B, C, n), dtype=grad_y.dtype, device=grad_y.device)
    return out.scatter_add_(2, _expand_index(indices.reshape(B, M * U), C), grad_y.reshape(B, C, M * U))
