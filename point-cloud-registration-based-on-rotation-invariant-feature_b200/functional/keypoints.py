"""compute_iss_keypoints / keypoint_batch — Intrinsic Shape Signatures keypoints (Zhong, ICCV Workshops 2009) on the GPU:
Open3D's `geometry.keypoint.compute_iss_keypoints`, every cloud of a batch in one call (csrc/iss.cu), and the bridge from
the keypoints to the batched matcher and pose solvers."""
import torch

from ..backend import _backend

__all__ = ['compute_iss_keypoints', 'keypoint_batch']


def compute_iss_keypoints(xyz, salient_radius=0.0, non_max_radius=0.0, gamma_21=0.975, gamma_32=0.975, min_neighbors=5,
                          return_saliency=False, return_radii=False):
    """xyz FloatTensor[B,3,N] (CUDA) -> (idx IntTensor[B,N], count IntTensor[B]).

    Open3D's names and defaults.  Point q is a keypoint when its neighbourhood within salient_radius (at least
    min_neighbors points, q included) has covariance eigenvalues e1 >= e2 >= e3 with e2/e1 < gamma_21 and e3/e2 < gamma_32,
    and its saliency e3 is positive and not exceeded within non_max_radius (which must hold min_neighbors points too).
    A radius of 0 sets both radii from the cloud's resolution r (the mean distance to the nearest other point): 6 r and
    4 r, computed per cloud on the device.  Points with a non-finite coordinate are ignored.

    Row b of idx lists the keypoints in ascending index in idx[b, :count[b]] and -1 after them.  return_saliency adds
    DoubleTensor[B,N] (e3 where the eigenvalue tests pass, else 0); return_radii adds FloatTensor[B,2] (salient, non-max)
    as used.  Extra outputs come back in that order.  include/ri_b200.h (ri_iss_keypoints_f32) states the arithmetic and
    the deltas from Open3D.  Not differentiable."""
    xyz = xyz.float().contiguous()
    idx, count, sal, radii = torch.ops.ri.iss_keypoints(xyz, float(salient_radius), float(non_max_radius),
                                                        float(gamma_21), float(gamma_32), int(min_neighbors),
                                                        bool(return_saliency))
    return (idx, count) + ((sal,) if return_saliency else ()) + ((radii,) if return_radii else ())


def keypoint_batch(xyz, idx, count, features=None):
    """Keypoints of a dense batch -> one fixed-size, point-major batch for matcher.mutual_nn and the pose solvers.

    xyz FloatTensor[B,3,N] and (idx, count) as compute_iss_keypoints returns them; features FloatTensor[B,C,N]
    (channel-major, e.g. compute_fpfh_feature of the full clouds) or None.  K = max(count, 1) is read with one host
    synchronisation.  Returns (points [B,K,3], features [B,K,C] or None, idx [B,K] int32), the layout of
    farthest_point_batch.

    Rows past count[b] repeat the cloud's FIRST keypoint.  The matcher breaks ties to the lowest index, so a padded row never
    wins a nearest-neighbour search against row 0 and can never form a mutual match: the padding leaves every match of the
    pair unchanged.  A cloud with no keypoints gets K copies of its point 0, which may still match; such a pair carries
    count[b] == 0 and its result should be discarded."""
    if xyz.dim() != 3 or xyz.shape[1] != 3:
        raise RuntimeError("xyz must be [B, 3, N]")
    B, _, N = xyz.shape
    if tuple(idx.shape) != (B, N) or tuple(count.shape) != (B,):
        raise RuntimeError("idx must be [B, N] and count [B], as compute_iss_keypoints returns them")
    if N == 0:
        raise RuntimeError("keypoint_batch needs clouds with at least one point")
    if features is not None and (features.dim() != 3 or features.shape[0] != B or features.shape[2] != N):
        raise RuntimeError("features must be [B, C, N]")
    K = max(int(count.max()) if B else 0, 1)
    cnt = count.to(torch.int32)
    row = torch.arange(K, device=xyz.device, dtype=torch.int32)[None, :]
    first = torch.where(cnt > 0, idx[:, 0].to(torch.int32), torch.zeros_like(cnt))
    sel = torch.where(row < cnt[:, None], idx[:, :K].to(torch.int32), first[:, None]).contiguous()
    points = _backend.gather_features_forward(xyz.float().contiguous(), sel).transpose(1, 2).contiguous()
    feats = None
    if features is not None:
        feats = _backend.gather_features_forward(features.float().contiguous(), sel).transpose(1, 2).contiguous()
    return points, feats, sel
