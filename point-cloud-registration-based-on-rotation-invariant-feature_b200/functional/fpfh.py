"""compute_fpfh_feature — FPFH descriptors (Rusu, Blodow, Beetz, ICRA 2009) of xyz + normal clouds on the GPU: Open3D's
`compute_fpfh_feature` with the hybrid (radius, max_nn) search, every cloud of a batch in one call (csrc/fpfh.cu)."""
import torch

__all__ = ['compute_fpfh_feature']


def compute_fpfh_feature(xyz, normals, radius, max_nn=100, return_counts=False, return_spfh=False):
    """xyz, normals FloatTensor[B,3,N] (CUDA; normals used as given, e.g. from estimate_normals) -> fpfh FloatTensor[B,33,N].

    Each point's neighbours are the `max_nn` nearest points (itself included, ties to the lower index) closer than
    `radius` (strict; radius=float('inf') gives the plain k-NN), 1 <= max_nn <= 128: the list estimate_normals uses.
    The 33 channels are Open3D's three 11-bin histograms (angle, v.n2, dp.n1).  A point with at most one neighbour gets
    zeros.  include/ri_b200.h (ri_compute_fpfh_f32) states the arithmetic and the deltas from Open3D.

    The output is channel-major [B,33,N], the layout matcher.mutual_nn and registration.register_pairs take.
    return_counts adds counts IntTensor[B,N] (list lengths); return_spfh adds the simplified histograms FloatTensor[B,33,N]
    (bin counts times 100 / (n - 1)).  Extra outputs come back in that order after fpfh.  Not differentiable."""
    xyz = xyz.float().contiguous()
    normals = normals.float().contiguous()
    fpfh, spfh, counts = torch.ops.ri.compute_fpfh(xyz, normals, float(radius), int(max_nn), bool(return_spfh),
                                                   bool(return_counts))
    out = (fpfh,) + ((counts,) if return_counts else ()) + ((spfh,) if return_spfh else ())
    return out if len(out) > 1 else fpfh
