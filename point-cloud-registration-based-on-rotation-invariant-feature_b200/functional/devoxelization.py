"""trilinear_devoxelize / spherical_trilinear_devoxelize — same contracts as
/root/reference/PVCNN/modules/functional/devoxelization.py:10-45 and spherical_devox.py:10-45."""
from torch.autograd import Function

from ..backend import _backend

__all__ = ['trilinear_devoxelize', 'spherical_trilinear_devoxelize']


class TrilinearDevoxelization(Function):
    """(features [B,C,r,r,r], coords [B,3,N] in grid units, r, is_training=True) -> [B,C,N]"""

    @staticmethod
    def forward(ctx, features, coords, resolution, is_training=True):
        B, C = features.shape[:2]
        outs, inds, wgts = _backend.trilinear_devoxelize_forward(resolution, is_training, coords.contiguous(),
                                                                 features.contiguous().view(B, C, -1))
        ctx.save_for_backward(inds, wgts)
        ctx.r = resolution
        return outs

    @staticmethod
    def backward(ctx, grad_output):
        inds, wgts = ctx.saved_tensors
        g = _backend.trilinear_devoxelize_backward(grad_output.contiguous(), inds, wgts, ctx.r)
        return g.view(grad_output.size(0), grad_output.size(1), ctx.r, ctx.r, ctx.r), None, None, None


class SphericalTrilinearDevoxelization(Function):
    """(features [B,C,r,r,r], normalised coords [B,3,N], g_inds [B,N], r >= 4, is_training=True) -> [B,C,N]"""

    @staticmethod
    def forward(ctx, features, coords, g_inds, resolution, is_training=True):
        B, C = features.shape[:2]
        outs, inds, wgts = _backend.spherical_trilinear_devoxelize_forward(
            resolution, is_training, coords.contiguous(), features.contiguous().view(B, C, -1), g_inds)
        ctx.save_for_backward(inds, wgts)
        ctx.r = resolution
        return outs

    @staticmethod
    def backward(ctx, grad_output):
        inds, wgts = ctx.saved_tensors
        g = _backend.spherical_trilinear_devoxelize_backward(grad_output.contiguous(), inds, wgts, ctx.r)
        return g.view(grad_output.size(0), grad_output.size(1), ctx.r, ctx.r, ctx.r), None, None, None, None


trilinear_devoxelize = TrilinearDevoxelization.apply
spherical_trilinear_devoxelize = SphericalTrilinearDevoxelization.apply
