"""The front end's backward pass on the GPU against the fp64 restatements of tests/grad_oracle.py.

  kernels      csrc/grad.cu (k-NN, voxelize, devoxelize backward) and the grouping backward of csrc/ballquery.cu, through
               torch.ops.ri.*, at full, odd and contended shapes: the voxelize backward is a pure gather and equals the C
               oracle bit for bit; the scatters use float atomics and must sit within TOL (max |d| / max |fp64|) of fp64.
  autograd     every torch.autograd.Function of functional/ against fp64 autograd of the restated forward, fed the
               indices and weights of our own forward (the forward tests pin those), with dense, summed (stride 0),
               expanded, permuted and sliced output gradients, and with only one output of a multi-output op in use.
  module       PVConv in train mode: its gradients are as close to an all-fp64 restatement as torch's own fp32 layers are.
The bar is the suite's TOL throughout; a gradient that misses it is a bug to fix, not a tolerance to widen."""
import copy

import numpy as np
import pytest
import torch

import grad_oracle as go
from _util import TOL

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def ri():
    import ri_b200
    return ri_b200


def gen(seed):
    return torch.Generator().manual_seed(seed)


def randn(g, *shape):
    return torch.randn(*shape, generator=g).to(DEV)


def d64(t):
    return t.detach().double()


def A(t):
    return t.detach().cpu().numpy()


def err(got, want):
    """max |got - want| / max |want| (the suite's scaled error), computed on the device in fp64."""
    if want.numel() == 0:
        return 0.0
    return float((got.double() - want.double()).abs().max() / want.double().abs().max().clamp_min(1e-30))


def sph_coords(g, B, N):
    """Normalised coordinates in the unit ball; the first points of each cloud are ones the spherical grid leaves undefined
    (ind = -1): the origin, the south-pole direction (beta = pi), radius exactly 1 and radius > 1."""
    v = torch.randn(B, 3, N, generator=g, dtype=torch.float64)
    v = v / v.norm(dim=1, keepdim=True) * torch.rand(B, 1, N, generator=g, dtype=torch.float64) ** (1 / 3)
    special = torch.tensor([[0.0, 0.0, 0.0], [0.0, 0.0, -0.5], [1.0, 0.0, 0.0], [0.0, 1.5, 0.0]], dtype=torch.float64).T
    q = min(N, 4)
    v[:, :, :q] = special[:, :q]
    return v.float().to(DEV).contiguous()


def cube_coords(g, B, N, r):
    """Grid-unit coordinates in [0, r-1] with points on cell faces (integer coordinates: the high corners get weight 0),
    on the far faces (r - 1) and at the grid's corners."""
    nc = torch.rand(B, 3, N, generator=g) * (r - 1)
    nc[:, :, :N // 8] = torch.round(nc[:, :, :N // 8])
    nc[:, 0, N // 8:N // 6] = r - 1
    nc[:, :, N // 6:N // 5] = torch.randint(0, 2, (B, 3, N // 5 - N // 6), generator=g).float() * (r - 1)
    return nc.to(DEV).contiguous()


# ===================================================================================== voxelize / devoxelize kernels
def _vox_devox_backward(ri, oracle, shape, nc, feat, r, g):
    B, C, N = feat.shape
    s = r ** 3
    sph = shape == "spherical"
    if sph:
        _, ind, cnt = torch.ops.ri.sph_voxelize(feat, nc, r)
    else:
        _, ind, cnt = torch.ops.ri.cube_voxelize(feat, torch.round(nc).to(torch.int32).contiguous(), r)
    gy = randn(g, B, C, s)
    gx = torch.ops.ri.voxelize_backward(gy, ind, cnt)
    assert torch.equal(gx, torch.ops.ri.voxelize_backward(gy, ind, cnt)), "voxelize backward is not deterministic"
    assert np.array_equal(A(gx), oracle.avg_voxelize_grad(A(gy), A(ind), A(cnt)))
    assert err(gx, go.avg_voxelize_grad(d64(gy), ind, cnt)) <= TOL
    grid = randn(g, B, C, s)
    if sph:
        _, inds, wgts = torch.ops.ri.sph_trilinear_devox(nc, grid, ind, r)
    else:
        _, inds, wgts = torch.ops.ri.trilinear_devox(nc, grid, r)
    gyd = randn(g, B, C, N)
    gxd = torch.ops.ri.devox_backward(gyd, inds, wgts, r, sph)
    e = err(gxd, go.devox_grad(d64(gyd), inds, wgts, s, sph))
    assert e <= TOL, e
    return ind


@pytest.mark.parametrize("shape,B,N,C,r", [
    ("spherical", 32, 1024, 67, 32), ("spherical", 1, 50000, 7, 64), ("spherical", 32, 777, 1, 4),
    ("spherical", 3, 777, 67, 5), ("spherical", 2, 1, 7, 5),
    ("cube", 32, 1024, 7, 32), ("cube", 1, 50000, 67, 64), ("cube", 2, 777, 67, 2), ("cube", 4, 1024, 67, 8),
    ("cube", 32, 1, 1, 8)])
def test_voxelize_and_devox_backward_kernels(ri, oracle, shape, B, N, C, r):
    """C = 7 and 67 leave a partial 8-channel group; B = 32 is the batch the front end runs; r = 64 and N = 50 000 are
    the largest grids and clouds; N = 1 a cloud of one point."""
    g = gen(1000 * r + N + C)
    nc = sph_coords(g, B, N) if shape == "spherical" else cube_coords(g, B, N, r)
    ind = _vox_devox_backward(ri, oracle, shape, nc, randn(g, B, C, N), r, g)
    if shape == "spherical":
        assert bool((ind == -1).any()), "the input must contain points the spherical grid leaves undefined"


@pytest.mark.parametrize("shape", ["spherical", "cube"])
def test_voxelize_and_devox_backward_under_contention(ri, oracle, shape):
    """Every point of a cloud in one cell (cloud 0: one location inside a cell, all 8 corners shared by all points; cloud 1:
    one grid node, all weight on a single corner): 4096-way float atomics on the same addresses."""
    B, N, C, r = 2, 4096, 9, 8
    g = gen(5)
    if shape == "spherical":
        nc = torch.empty(B, 3, N, device=DEV)
        nc[0] = torch.tensor([0.31, 0.22, 0.13], device=DEV)[:, None]
        nc[1] = torch.tensor([0.0, 0.6, 0.0], device=DEV)[:, None]
    else:
        nc = torch.empty(B, 3, N, device=DEV)
        nc[0] = torch.tensor([3.5, 2.25, 6.75], device=DEV)[:, None]
        nc[1] = float(r - 1)
    ind = _vox_devox_backward(ri, oracle, shape, nc.contiguous(), randn(g, B, C, N), r, g)
    assert bool((ind == ind[:, :1]).all())


def test_spherical_devox_refuses_r_below_4(ri, oracle):
    """Below r = 4 the spherical corner indices (up to r^2 + 7r + 4) leave the r^3 grid: the op raises before it launches
    anything.  The cell indices come from the C oracle, which shows they stay inside the grid."""
    g = gen(9)
    B, N, C = 2, 300, 5
    nc = sph_coords(g, B, N)
    for r in (2, 3):
        ind, _ = oracle.sph_grid_stats(A(nc), r)
        assert ind.max() < r ** 3
        ind = torch.from_numpy(ind).to(DEV)
        grid = randn(g, B, C, r, r, r)
        with pytest.raises(RuntimeError):
            torch.ops.ri.sph_trilinear_devox(nc, grid.view(B, C, -1), ind, r)
        with pytest.raises(RuntimeError):
            ri.functional.spherical_trilinear_devoxelize(grid, nc, ind, r, True)
    torch.cuda.synchronize()


# ============================================================================================== k-NN kernel
@pytest.mark.parametrize("B,c,n,m,k", [(32, 3, 1024, 1024, 20), (1, 3, 50000, 1024, 32), (3, 5, 777, 300, 16),
                                        (2, 1, 777, 1024, 1), (4, 3, 1024, 777, 32)])
def test_knn_backward_kernel(ri, B, c, n, m, k):
    g = gen(n + m + k)
    x1, x2 = randn(g, B, c, n), randn(g, B, c, m)
    x2[:, :, -3:] = x2[:, :, :3]                                          # duplicated references
    _, _, i1, i2 = torch.ops.ri.knn(x1, x2, k)
    gd1, gd2 = randn(g, B, k, n), randn(g, B, k, m)
    got = torch.ops.ri.knn_backward(x1, x2, gd1, gd2, i1, i2)
    want = go.knn_grad(d64(x1), d64(x2), d64(gd1), d64(gd2), i1, i2)
    for a, b in zip(got, want):
        e = err(a, b)
        assert e <= TOL, e


def test_knn_backward_sentinels_and_skip_rule(ri):
    """m < k and queries farther than 100 units from every reference: their slots hold the forward's sentinel (10000,
    index 0) and still push 2g (x - ref_0) onto reference point 0; a slot whose 2 * graddist >= 20000 adds nothing."""
    g = gen(17)
    B, c, n, m, k = 2, 3, 200, 5, 8
    x1, x2 = randn(g, B, c, n), randn(g, B, c, m)
    x1[:, 0, :4] += 150.0
    d1, d2, i1, i2 = torch.ops.ri.knn(x1, x2, k)
    assert bool((d1[:, :, :4] == 10000).all()) and bool((i1[:, :, :4] == 0).all())
    assert bool((d1[:, m:] == 10000).all())
    gd1, gd2 = randn(g, B, k, n), randn(g, B, k, m)
    gd1[:, 0, 4:8] = 10000.0                                              # skipped
    gd1[:, 1, 4:8] = 9999.0                                               # kept
    gd1[:, 2, 8:12] = 25000.0                                             # skipped
    got = torch.ops.ri.knn_backward(x1, x2, gd1, gd2, i1, i2)
    want = go.knn_grad(d64(x1), d64(x2), d64(gd1), d64(gd2), i1, i2)
    for a, b in zip(got, want):
        e = err(a, b)
        assert e <= TOL, e


def test_knn_backward_one_reference_for_every_query(ri):
    """One reference is the nearest neighbour of all 4096 queries: 4096-way float atomics onto one point."""
    g = gen(23)
    B, n, m, k = 2, 4096, 64, 1
    x2 = randn(g, B, 3, m)
    x2 = x2 / x2.norm(dim=1, keepdim=True) * 40.0
    x2[:, :, 0] = 0.0
    x1 = randn(g, B, 3, n) * 0.5 + 0.25
    _, _, i1, i2 = torch.ops.ri.knn(x1, x2.contiguous(), k)
    assert bool((i1 == 0).all())
    gd1, gd2 = randn(g, B, k, n), randn(g, B, k, m)
    got = torch.ops.ri.knn_backward(x1, x2.contiguous(), gd1, gd2, i1, i2)
    want = go.knn_grad(d64(x1), d64(x2), d64(gd1), d64(gd2), i1, i2)
    for a, b in zip(got, want):
        e = err(a, b)
        assert e <= TOL, e


# ========================================================================================== grouping kernel
@pytest.mark.parametrize("B,C,N,M,U", [(2, 67, 1024, 1024, 128), (3, 7, 777, 300, 16)])
def test_grouping_backward_kernel(ri, B, C, N, M, U):
    g = gen(N + U)
    pts = randn(g, B, 3, N) * 0.5
    idx = torch.ops.ri.ball_query(pts[:, :, :M].contiguous(), pts, 0.3, U)   # first hit replicated: repeated indices
    gy = randn(g, B, C, M, U)
    got = torch.ops.ri.grouping_backward(gy, idx, N)
    e = err(got, go.grouping_grad(d64(gy), idx, N))
    assert e <= TOL, e


# ============================================================================================ autograd wiring
B_, C_, N_, R_ = 3, 13, 600, 8


def _case(ri, name, g):
    """-> (leaves, index of each leaf that must get no gradient, ours(*leaves) -> outputs, ref(*fp64 leaves) -> outputs).
    `ref` reuses the indices and weights our forward produced; only the differentiable arithmetic is restated."""
    F, ops = ri.functional, torch.ops.ri
    B, C, N, r = B_, C_, N_, R_
    s = r ** 3
    feat = randn(g, B, C, N).requires_grad_(True)
    if name == "knn":
        x1, x2 = randn(g, B, 3, N).requires_grad_(True), randn(g, B, 3, 450).requires_grad_(True)
        _, _, i1, i2 = ops.knn(x1.detach(), x2.detach(), 8)
        return [x1, x2], [], lambda a, b: F.k_nearest_neighbor(a, b, 8)[:2], lambda a, b: go.knn_dist(a, b, i1, i2)
    if name in ("avg_vox", "avg_vox_edge"):
        vox = torch.randint(0, r, (B, 3, N), generator=g, dtype=torch.int32).to(DEV)
        ind = ops.cube_voxelize(feat.detach(), vox, r)[1]
        fn = F.avg_voxelize if name == "avg_vox" else F.avg_voxelize_edge
        ours = lambda f: tuple(o for o in fn(f, vox, r) if o.is_floating_point())
        return [feat], [], ours, _restated_vox(ind, r, name.endswith("edge"))
    if name in ("sph_avg_vox", "sph_avg_vox_edge"):
        nc = sph_coords(g, B, N).requires_grad_(True)
        ind = ops.sph_voxelize(feat.detach(), nc.detach(), r)[1]
        assert bool((ind == -1).any())
        fn = F.spherical_avg_voxelize if name == "sph_avg_vox" else F.spherical_avg_voxelize_edge
        ours = lambda f, c: tuple(o for o in fn(f, c, r) if o.is_floating_point())
        vox = _restated_vox(ind, r, name.endswith("edge"))
        return [feat, nc], [1], ours, lambda f, c: vox(f)
    if name == "devox":
        grid = randn(g, B, C, r, r, r).requires_grad_(True)
        nc = cube_coords(g, B, N, r).requires_grad_(True)
        _, inds, wgts = ops.trilinear_devox(nc.detach(), grid.detach().view(B, C, s), r)
        return ([grid, nc], [1], lambda v, c: (F.trilinear_devoxelize(v, c, r, True),),
                lambda v, c: (go.devox(v, inds, wgts),))
    if name == "sph_devox":
        grid = randn(g, B, C, r, r, r).requires_grad_(True)
        nc = sph_coords(g, B, N).requires_grad_(True)
        ind = ops.sph_voxelize(feat.detach(), nc.detach(), r)[1]
        _, inds, wgts = ops.sph_trilinear_devox(nc.detach(), grid.detach().view(B, C, s), ind, r)
        return ([grid, nc], [1], lambda v, c: (F.spherical_trilinear_devoxelize(v, c, ind, r, True),),
                lambda v, c: (go.devox(v, inds, wgts),))
    if name == "edge":
        avg = randn(g, B, C, r, r, r).requires_grad_(True)
        ind = ops.sph_voxelize(feat.detach(), sph_coords(g, B, N), r)[1]
        assert bool((ind == -1).any())
        return ([avg, feat], [], lambda a, f: (F.voxel_edge_features(a, f, ind),),
                lambda a, f: (go.voxel_edge_features(a, f, ind),))
    if name == "grouping":
        pts = randn(g, B, 3, N) * 0.5
        idx = ops.ball_query(pts[:, :, :200].contiguous(), pts, 0.3, 32)
        return [feat], [], lambda f: (F.grouping(f, idx),), lambda f: (go.grouping(f, idx),)
    raise ValueError(name)


def _restated_vox(ind, r, edge):
    def ref(f):
        B, C = f.shape[:2]
        grid = go.avg_voxelize(f, ind, r ** 3)
        outs = (grid.view(B, C, r, r, r),)
        return outs + (go.voxel_edge_features(grid, f, ind),) if edge else outs
    return ref


def _grad_outputs(g, outs, mode):
    Ws = []
    for o in outs:
        shape = tuple(o.shape)
        if mode == "dense":
            w = randn(g, *shape)
        elif mode == "expanded":                                          # stride 0 along the last axis
            w = randn(g, *shape[:-1], 1).expand(shape)
        elif mode == "permuted":
            w = randn(g, *shape[::-1]).permute(*range(len(shape) - 1, -1, -1))
        elif mode == "slice":
            w = randn(g, *shape[:-1], 2 * shape[-1] + 1)[..., 1::2]
        else:
            raise ValueError(mode)
        assert tuple(w.shape) == shape
        Ws.append(w)
    return Ws


FUNCTIONS = ["knn", "avg_vox", "sph_avg_vox", "avg_vox_edge", "sph_avg_vox_edge", "devox", "sph_devox", "edge", "grouping"]
MULTI_OUTPUT = ["knn", "avg_vox_edge", "sph_avg_vox_edge"]


@pytest.mark.parametrize("name,mode", [(n, m) for n in FUNCTIONS for m in ("dense", "sum", "expanded", "permuted", "slice")] +
                         [(n, m) for n in MULTI_OUTPUT for m in ("first_only", "last_only")])
def test_function_gradients_match_fp64_autograd(ri, name, mode):
    """`sum` differentiates out.sum() (the output gradient arrives expanded, stride 0 everywhere); first_only / last_only use
    one output of a multi-output op (dist1 or dist2; the grid or the edge features) and leave the other's gradient to
    autograd's zeros.  Coordinates get no gradient, as in the reference."""
    g = gen(FUNCTIONS.index(name) * 10 + len(mode))
    leaves, no_grad, ours, ref = _case(ri, name, g)
    outs = ours(*leaves)
    leaves64 = [d64(x).requires_grad_(True) for x in leaves]
    outs64 = ref(*leaves64)
    assert len(outs) == len(outs64) and all(a.shape == b.shape for a, b in zip(outs, outs64))
    if mode in ("first_only", "last_only"):
        pick = 0 if mode == "first_only" else -1
        outs, outs64 = (outs[pick],), (outs64[pick],)
    if mode == "sum":
        got = torch.autograd.grad(sum(o.sum() for o in outs), leaves, allow_unused=True)
        want = torch.autograd.grad(sum(o.sum() for o in outs64), leaves64, allow_unused=True)
    else:
        Ws = _grad_outputs(g, outs, "dense" if mode.endswith("_only") else mode)
        got = torch.autograd.grad(outs, leaves, Ws, allow_unused=True)
        want = torch.autograd.grad(outs64, leaves64, [w.double() for w in Ws], allow_unused=True)
    for j, (a, b) in enumerate(zip(got, want)):
        if j in no_grad:
            assert a is None, "input %d must not receive a gradient" % j
            continue
        assert a is not None and b is not None and a.shape == b.shape
        assert float(b.abs().max()) > 0
        e = err(a, b)
        assert e <= TOL, (j, e)


# ================================================================================================ PVConv module
def _restate_functional(ri, mp):
    """Point ri_b200.functional's voxelize / devoxelize ops at the restatements (in the dtype of the features), indices and
    corner weights from our own forward on the same fp32 coordinates."""
    F, ops = ri.functional, torch.ops.ri

    def vox(features, coords, r, sph, edge):
        f32 = features.detach().float().contiguous()
        if sph:
            ind = ops.sph_voxelize(f32, coords.float().contiguous(), r)[1]
        else:
            ind = ops.cube_voxelize(f32, coords.int().contiguous(), r)[1]
        outs = _restated_vox(ind, r, edge)(features)
        return (outs[0], ind) + outs[1:]

    def devox(features, coords, r, is_training=True):
        B, C = features.shape[:2]
        g32 = features.detach().float().reshape(B, C, -1).contiguous()
        _, inds, wgts = ops.trilinear_devox(coords.float().contiguous(), g32, r)
        return go.devox(features, inds, wgts)

    def sph_devox(features, coords, g_inds, r, is_training=True):
        B, C = features.shape[:2]
        g32 = features.detach().float().reshape(B, C, -1).contiguous()
        _, inds, wgts = ops.sph_trilinear_devox(coords.float().contiguous(), g32, g_inds, r)
        return go.devox(features, inds, wgts)

    mp.setattr(F, "avg_voxelize", lambda f, c, r: vox(f, c, r, False, False))
    mp.setattr(F, "avg_voxelize_edge", lambda f, c, r: vox(f, c, r, False, True))
    mp.setattr(F, "spherical_avg_voxelize", lambda f, c, r: vox(f, c, r, True, False))
    mp.setattr(F, "spherical_avg_voxelize_edge", lambda f, c, r: vox(f, c, r, True, True))
    mp.setattr(F, "trilinear_devoxelize", devox)
    mp.setattr(F, "spherical_trilinear_devoxelize", sph_devox)


@pytest.mark.parametrize("kernel", ["dgcnn_kernel", "pointnet_kernel"])
@pytest.mark.parametrize("shape", ["spherical", "cube"])
def test_pvconv_gradients_as_close_to_fp64_as_torch_layers(ri, monkeypatch, shape, kernel):
    """PVConv (with_se, with_coeff, train mode, TF32 off) three times on the same weights and inputs: with our ops (fp32),
    with the ops restated in torch (fp32), and all in fp64 with the restated ops.  Every parameter and input gradient of ours
    is as close to fp64 as the torch-restated fp32 run is (the bar of the fused local-feature branch test)."""
    from ri_b200 import synth
    torch.manual_seed(3)
    B, N, C, Co, r = 2, 1024, 13, 24, 8
    base = ri.modules.PVConv(C, Co, kernel, shape, 3, r, with_coeff=True, with_se=True, normalize=False)
    with torch.no_grad():
        base.coefficient.fill_(0.7)
    coords = torch.from_numpy(synth.make_clouds(B, N, seed=91)[:, :3].copy()).to(DEV)
    g = gen(91)
    feat, W = randn(g, B, C, N), randn(g, B, Co, N)

    def run(dtype, restated):
        m = copy.deepcopy(base).to(device=DEV, dtype=dtype).train()
        x = feat.to(dtype).requires_grad_(True)
        with monkeypatch.context() as mp:
            if restated:
                _restate_functional(ri, mp)
            out, _ = m((x, coords))
        return torch.autograd.grad((out * W.to(dtype)).sum(), [x] + list(m.parameters()))

    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ours, t32, ref = run(torch.float32, False), run(torch.float32, True), run(torch.float64, True)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    names = ["features"] + [n for n, _ in base.named_parameters()]
    for name, a, t, w in zip(names, ours, t32, ref):
        e_ours, e_torch = err(a, w), err(t, w)
        assert e_ours <= max(4 * e_torch, 2e-6), (name, e_ours, e_torch)
