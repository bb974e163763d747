"""gather / furthest_point_sample — the contracts of the reference's functional/sampling.py (F.gather,
F.furthest_point_sample; backend sampling/sampling.cu), served by csrc/fps.cu and the grouping kernels (SURVEY.md §8f
row f12)."""
import torch

from ..backend import _backend

__all__ = ['gather', 'furthest_point_sample']


class Gather(torch.autograd.Function):
    """features FloatTensor[B,C,N], indices IntTensor[B,M] -> FloatTensor[B,C,M]; the backward sums the gradients of
    repeated indices."""

    @staticmethod
    def forward(ctx, features, indices):
        features = features.contiguous()
        indices = indices.int().contiguous()
        ctx.save_for_backward(indices)
        ctx.num_points = features.size(-1)
        return _backend.gather_features_forward(features, indices)

    @staticmethod
    def backward(ctx, grad_output):
        indices, = ctx.saved_tensors
        return _backend.gather_features_backward(grad_output.contiguous(), indices, ctx.num_points), None


gather = Gather.apply


def furthest_point_sample(coords, num_samples, lengths=None, return_indices=False):
    """coords FloatTensor[B,3,N] (CUDA) -> the sampled coordinates FloatTensor[B,3,num_samples] (the reference's return
    value), and their indices IntTensor[B,num_samples] too with return_indices=True.

    Cloud b uses its first lengths[b] points (a list or a CPU tensor, 0 <= lengths[b] <= N; None: all N).  Sampling starts
    at index 0 and takes the point farthest (fp64 squared distance) from those taken so far, the lowest index on ties;
    once every distinct point is taken the last index repeats, and an empty cloud gives indices -1 (and its gathered
    coordinates are then undefined).  At most 131072 points per cloud."""
    coords = coords.float().contiguous()
    if lengths is not None:
        lengths = torch.as_tensor(lengths, dtype=torch.int32, device="cpu")
    idx = torch.ops.ri.furthest_point_sample(coords, lengths, int(num_samples))
    empty_possible = lengths is not None or coords.shape[-1] == 0
    out = gather(coords, idx.clamp(min=0) if empty_possible else idx)
    return (out, idx) if return_indices else out
