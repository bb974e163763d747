"""estimate_normals — per-point normals of xyz-only clouds on the GPU: Open3D's `estimate_normals` with the hybrid
(radius, max_nn) search and its camera orientation, which the reference runs on the host (utils/open3d_func.py:77-83)."""
import torch

__all__ = ['estimate_normals']


def estimate_normals(xyz, radius, max_nn=30, camera=None, prior=None, return_counts=False):
    """xyz FloatTensor[B,3,N] (CUDA) -> normals FloatTensor[B,3,N] (and counts IntTensor[B,N] with return_counts=True).

    Each point's neighbours are the `max_nn` nearest points (itself included, ties to the lower index) closer than
    `radius` (strict; radius=float('inf') gives the plain k-NN), 1 <= max_nn <= 32.  The normal is the unit eigenvector
    of the smallest eigenvalue of their population covariance, computed in fp64; a point with fewer than 3 neighbours,
    or whose neighbours all coincide, gets (0, 0, 1).

    Orientation, at most one of:
      camera  FloatTensor[3] (shared) or [B,3]: each normal is flipped to face the camera, n.(camera - p) >= 0
              (Open3D's orient_normals_towards_camera_location);
      prior   FloatTensor[B,3,N]: each normal is flipped to agree with the prior, n.prior >= 0.
    Without either the sign is the solver's: deterministic, but arbitrary.

    counts: the number of neighbours each normal was fitted to.  The normals are not differentiable (no backward)."""
    xyz = xyz.float().contiguous()
    if camera is not None:
        camera = camera.float()
        if camera.dim() == 1 and xyz.dim() == 3:
            camera = camera.expand(xyz.shape[0], -1)
        camera = camera.contiguous()
    if prior is not None:
        prior = prior.float().contiguous()
    normals, counts = torch.ops.ri.estimate_normals(xyz, float(radius), int(max_nn), camera, prior)
    return (normals, counts) if return_counts else normals
