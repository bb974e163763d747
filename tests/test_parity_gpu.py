"""GPU parity tests: the sm_100a kernels (through torch.ops.ri.* -> the C ABI) against
  (1) what the reference's own CUDA kernels return on the same inputs, for every output compared bit for bit
      (tests/golden/reference_outputs.npz, the `reference` fixture; inputs regenerated from their seeds),
  (2) the committed golden vectors those kernels produced on adversarial inputs (tests/golden/),
  (3) the CPU oracle (oracle/ri_oracle.c).
Bar (north_star): voxel indices, counts, KNN indices (full order), devox corner indices bit-exact; PPF, voxel means,
devoxelized features, distances within 1e-5 relative (fp32)."""
import numpy as np
import pytest
import torch

from _util import TOL, load_golden, rel_err, scaled_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ri():
    import ri_b200
    return ri_b200


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def randn(seed, *shape):
    """Seeded standard-normal float32 on the device (numpy's generator: the same values on every machine)."""
    return T(np.random.default_rng(seed).standard_normal(shape, dtype=np.float32))


def A(t):
    return t.detach().cpu().numpy()


def clouds(B, N, seed, surface=True):
    from ri_b200 import synth
    return synth.make_clouds(B, N, seed=seed) if surface else np.random.default_rng(seed).standard_normal((B, 6, N)).astype(np.float32)


def sph_norm(xyz):
    nc = xyz - xyz.mean(2, keepdim=True)
    return (nc / (nc.norm(dim=1, keepdim=True).max(dim=2, keepdim=True).values + 1e-20)).contiguous()


# ================================================================================================ KNN
def test_knn_golden(ri, golden_dir):
    g = load_golden(golden_dir, "knn.npz")
    d1, d2, i1, i2 = torch.ops.ri.knn(T(g["xyz1"]), T(g["xyz2"]), int(g["k"]))
    assert np.array_equal(A(i1), g["idx1"]) and np.array_equal(A(i2), g["idx2"])
    assert np.array_equal(A(d1), g["dist1"]) and np.array_equal(A(d2), g["dist2"])      # same fma chain -> same bits
    e = load_golden(golden_dir, "knn_edge.npz")
    d1, d2, i1, i2 = torch.ops.ri.knn(T(e["xq"]), T(e["xs"]), 8)                        # m < k
    assert np.array_equal(A(i1), e["idx1"]) and np.array_equal(A(i2), e["idx2"])
    assert np.array_equal(A(d1), e["dist1"]) and np.array_equal(A(d2), e["dist2"])
    d, i = torch.ops.ri.knn_one(T(e["xc"]), T(e["xc"]), 20)
    assert np.array_equal(A(i), e["self_idx"]) and np.array_equal(A(d), e["self_dist"])
    d1, d2, i1, i2 = torch.ops.ri.knn(T(e["x5"]), T(e["y5"]), 4)                        # generic channel count
    assert np.array_equal(A(i1), e["c5_idx1"]) and np.array_equal(A(i2), e["c5_idx2"])
    assert np.array_equal(A(d1), e["c5_dist1"]) and np.array_equal(A(d2), e["c5_dist2"])


@pytest.mark.parametrize("n,m,k", [(1024, 1024, 20), (1000, 777, 16), (33, 2100, 5), (512, 512, 32), (64, 64, 1),
                                    (300, 300, 40)])
def test_knn_vs_reference_and_oracle(ri, reference, oracle, n, m, k):
    B = 3
    x1 = clouds(B, n, 1)[:, :3].copy(); x2 = clouds(B, m, 2)[:, :3].copy()
    q = min(n, m) // 2
    x2[:, :, :q] = x1[:, :, :q]                       # shared points: d = 0 and ties
    x2[:, :, m - 4:] = x2[:, :, :4]                   # duplicates at the far end
    d1, d2, i1, i2 = torch.ops.ri.knn(T(x1), T(x2), k)
    reference.equal("knn/%d-%d-%d" % (n, m, k), {"idx1": i1, "idx2": i2, "dist1": d1, "dist2": d2},
                    lambda b: dict(zip(("dist1", "dist2", "idx1", "idx2"), b.knn_forward_cuda(T(x1), T(x2), k))))
    o1, o2, p1, p2 = oracle.knn(x1, x2, k)
    assert np.array_equal(A(i1), p1) and np.array_equal(A(i2), p2)
    assert np.array_equal(A(d1), o1) and np.array_equal(A(d2), o2)


def test_knn_full_size_properties(ri):
    """BASELINE size (32 x 1024, k = 20): size-independent properties."""
    x = T(clouds(32, 1024, 3)[:, :3].copy())
    d, i = torch.ops.ri.knn_one(x, x, 20)
    assert bool((d[:, 1:] >= d[:, :-1]).all())                         # ascending along k
    assert bool((d[:, 0] == 0).all())                                  # self (or an exact duplicate) first
    assert int(i.min()) >= 0 and int(i.max()) < 1024
    gathered = torch.gather(x, 2, i.reshape(32, 1, -1).expand(-1, 3, -1).long()).reshape(32, 3, 20, 1024)
    diff = x[:, :, None, :] - gathered
    d_re = torch.addcmul(torch.addcmul(diff[:, 0] * diff[:, 0], diff[:, 1], diff[:, 1]), diff[:, 2], diff[:, 2])
    assert float((d_re - d).abs().max()) <= 1e-6                       # indices really are at those distances
    full = ((x[:, :, :, None] - x[:, :, None, :]) ** 2).sum(1)
    kth = full.kthvalue(20, dim=2).values
    assert float((kth - d[:, 19]).abs().max()) <= 1e-5                 # k-th distance matches a dense reference
    d2, i2 = torch.ops.ri.knn_one(x, x, 20)
    assert torch.equal(i, i2)                                          # deterministic


def test_knn_backward(ri, golden_dir):
    g = load_golden(golden_dir, "knn.npz")
    g1, g2 = torch.ops.ri.knn_backward(T(g["xyz1"]), T(g["xyz2"]), T(g["graddist1"]), T(g["graddist2"]),
                                       T(g["idx1"]), T(g["idx2"]))
    assert scaled_err(A(g1), g["gradxyz1"]) <= TOL and scaled_err(A(g2), g["gradxyz2"]) <= TOL


def test_knn_ppf_fused_equals_two_kernels(ri):
    for B, N, k in [(4, 1024, 20), (3, 777, 16), (2, 2048, 32), (2, 40, 8), (1, 10, 20), (2, 3000, 20)]:
        pts = clouds(B, N, 21 + N)
        pts[:, :, N // 2:N // 2 + 3] = pts[:, :, :3]                  # duplicated points (ties) and ...
        pts[:, 3:, 5] = 0.0                                             # ... a zero normal (degenerate column)
        xyz, nrm = T(pts[:, :3].copy()), T(pts[:, 3:].copy())
        d0, i0 = torch.ops.ri.knn_one(xyz, xyz, k)
        p0 = torch.ops.ri.ppf_gather(xyz, nrm, i0)
        d1, i1, p1 = torch.ops.ri.knn_ppf(xyz, nrm, k)
        assert torch.equal(i0, i1) and torch.equal(d0, d1) and torch.equal(p0, p1)
        if N <= 2048 and k <= 32:                                       # the fused kernel itself, whatever the op dispatches to
            L = ri._lib
            d2 = torch.empty_like(d0); i2 = torch.empty_like(i0); p2 = torch.empty_like(p0)
            L.check(L.lib.ri_knn_ppf_f32(xyz.data_ptr(), nrm.data_ptr(), 3 * N, B, N, k, d2.data_ptr(), i2.data_ptr(),
                                         p2.data_ptr(), torch.cuda.current_stream().cuda_stream), "knn_ppf")
            assert torch.equal(i0, i2) and torch.equal(d0, d2) and torch.equal(p0, p2)
    # straight off the interleaved [B,6,N] batch (cloud stride 6N), as the front-end engine calls it
    pts = T(clouds(4, 1024, 5)); B, N, k = 4, 1024, 20
    L = ri._lib
    d = torch.empty((B, k, N), device="cuda"); i = torch.empty((B, k, N), dtype=torch.int32, device="cuda")
    o = torch.empty((B, 4, k, N), device="cuda")
    L.check(L.lib.ri_knn_ppf_f32(pts.data_ptr(), pts.data_ptr() + 3 * N * 4, 6 * N, B, N, k, d.data_ptr(), i.data_ptr(),
                                 o.data_ptr(), torch.cuda.current_stream().cuda_stream), "knn_ppf")
    d1, i1, p1 = torch.ops.ri.knn_ppf(pts[:, :3].contiguous(), pts[:, 3:].contiguous(), k)
    assert torch.equal(i, i1) and torch.equal(d, d1) and torch.equal(o, p1)


def test_split_and_packed_ppf(ri):
    L = ri._lib
    st = torch.cuda.current_stream().cuda_stream
    for B, N, k in [(4, 1024, 20), (3, 777, 7), (2, 50, 20)]:
        pts = T(clouds(B, N, 31 + N))
        xyz = torch.empty((B, 3, N), device="cuda"); nrm = torch.empty((B, 3, N), device="cuda")
        packed = torch.empty((B, N, 8), device="cuda")
        L.check(L.lib.ri_split_xyz_normals_f32(pts.data_ptr(), B, N, xyz.data_ptr(), nrm.data_ptr(), packed.data_ptr(), st), "split")
        assert torch.equal(xyz, pts[:, :3].contiguous()) and torch.equal(nrm, pts[:, 3:].contiguous())
        assert torch.equal(packed[:, :, :6], pts.permute(0, 2, 1).contiguous()) and bool((packed[:, :, 6:] == 0).all())
        _, idx = torch.ops.ri.knn_one(xyz, xyz, k)
        want = torch.ops.ri.ppf_gather(xyz, nrm, idx)
        got = torch.empty_like(want)
        L.check(L.lib.ri_ppf_gather_packed_f32(packed.data_ptr(), idx.data_ptr(), B, N, k, got.data_ptr(), st), "ppf_packed")
        assert torch.equal(got, want)


# ================================================================================================ PPF
def test_ppf_golden(ri, golden_dir, oracle):
    g = load_golden(golden_dir, "ppf.npz")
    f = torch.ops.ri.ppf(T(g["coords"]), T(g["center"]), T(g["normals"]), T(g["center_normal"]))
    assert rel_err(A(f), g["feat"]) <= TOL
    assert np.array_equal(A(f), g["feat"])           # same op order + same f64 acos => identical bits
    o = oracle.ppf_backend(g["coords"], g["center"], g["normals"], g["center_normal"])
    assert np.max(np.abs(o - g["feat"])) <= 1e-6      # host libm acos vs device acos: <= 1 ulp of pi


def test_ppf_gather_equals_columns(ri, reference):
    B, N, k = 4, 1024, 20
    pts = clouds(B, N, 5)
    xyz, nrm = T(pts[:, :3].copy()), T(pts[:, 3:].copy())
    _, idx = torch.ops.ri.knn_one(xyz, xyz, k)
    fused = torch.ops.ri.ppf_gather(xyz, nrm, idx)                                    # [B,4,k,N]
    gi = idx.reshape(B, 1, k * N).expand(-1, 3, -1).long()
    p_xyz, p_nrm = torch.gather(xyz, 2, gi), torch.gather(nrm, 2, gi)
    c_xyz = xyz[:, :, None, :].expand(-1, -1, k, -1).reshape(B, 3, k * N).contiguous()
    c_nrm = nrm[:, :, None, :].expand(-1, -1, k, -1).reshape(B, 3, k * N).contiguous()
    cols = ri.functional.ppf(c_xyz, p_xyz, c_nrm, p_nrm).reshape(B, 4, k, N)
    assert torch.equal(fused, cols)
    reference.equal("ppf_gather", {"": fused}, lambda b: {"": b.spherical_ppf_forward(
        p_xyz.contiguous(), c_xyz, p_nrm.contiguous(), c_nrm).reshape(B, 4, k, N)})
    # neighbour 0 is the point itself: direction undefined -> angles pi/2, ||d|| clamps to 1e-20
    assert float((fused[:, 3, 0] - 1e-20).abs().max()) < 1e-26
    assert float((fused[:, 0, 0] - np.pi / 2).abs().max()) < 1e-6


# ================================================================================================ voxelize
@pytest.mark.parametrize("r", [4, 8, 16, 32])
def test_sph_voxelize_golden(ri, golden_dir, r):
    g = load_golden(golden_dir, "spherical.npz")
    out, ind, cnt = torch.ops.ri.sph_voxelize(T(g[f"r{r}_feat"]), T(g[f"r{r}_coords"]), r)
    assert np.array_equal(A(ind), g[f"r{r}_ind"])
    assert np.array_equal(A(cnt), g[f"r{r}_cnt"])
    assert scaled_err(A(out), g[f"r{r}_out"]) <= TOL
    gx = torch.ops.ri.voxelize_backward(T(g[f"r{r}_gy"]), ind, cnt)
    assert rel_err(A(gx), g[f"r{r}_gx"]) <= TOL
    o, di, dw = torch.ops.ri.sph_trilinear_devox(T(g[f"r{r}_coords"]), T(g[f"r{r}_grid"]), ind, r)
    assert np.array_equal(A(di), g[f"r{r}_dinds"])
    assert np.array_equal(A(dw), g[f"r{r}_dwgts"])
    assert scaled_err(A(o), g[f"r{r}_douts"]) <= TOL
    dgx = torch.ops.ri.devox_backward(T(g[f"r{r}_dgy"]), di, dw, r, True)
    assert scaled_err(A(dgx), g[f"r{r}_dgx"]) <= TOL


@pytest.mark.parametrize("r", [4, 8, 16])
def test_cube_voxelize_golden(ri, golden_dir, r):
    g = load_golden(golden_dir, "cube.npz")
    out, ind, cnt = torch.ops.ri.cube_voxelize(T(g[f"r{r}_feat"]), T(g[f"r{r}_vox"]), r)
    assert np.array_equal(A(ind), g[f"r{r}_ind"]) and np.array_equal(A(cnt), g[f"r{r}_cnt"])
    assert scaled_err(A(out), g[f"r{r}_out"]) <= TOL
    gx = torch.ops.ri.voxelize_backward(T(g[f"r{r}_gy"]), ind, cnt)
    assert rel_err(A(gx), g[f"r{r}_gx"]) <= TOL
    o, di, dw = torch.ops.ri.trilinear_devox(T(g[f"r{r}_norm_coords"]), T(g[f"r{r}_grid"]), r)
    assert np.array_equal(A(di), g[f"r{r}_dinds"]) and np.array_equal(A(dw), g[f"r{r}_dwgts"])
    assert np.array_equal(A(o), g[f"r{r}_douts"])
    dgx = torch.ops.ri.devox_backward(T(g[f"r{r}_dgy"]), di, dw, r, False)
    assert scaled_err(A(dgx), g[f"r{r}_dgx"]) <= TOL


@pytest.mark.parametrize("B,N,C,r", [(32, 1024, 67, 32), (5, 1000, 9, 16), (3, 4096, 4, 64), (2, 777, 3, 8),
                                      (2, 6000, 3, 32), (2, 500, 3, 5), (1, 50000, 4, 64)])
def test_sph_voxelize_vs_reference(ri, reference, oracle, B, N, C, r):
    """Cell indices and counts against the reference kernels' at full and odd sizes; the means over the whole grid against the
    C oracle's mean of every cell over the points those indices put in it.  (N = 6000 / 50000 take the scan-sized sorted path,
    r = 5 the atomic fallback.)"""
    pts = clouds(B, N, 11 + r)
    nc = sph_norm(T(pts[:, :3].copy()))
    feat = randn([B, N, C, r], B, C, N)
    out, ind, cnt = torch.ops.ri.sph_voxelize(feat, nc, r)
    assert int(cnt.sum()) == int((ind >= 0).sum())
    reference.equal("sph_voxelize/%d-%d-%d-%d" % (B, N, C, r), {"ind": ind, "cnt": cnt},
                    lambda b: dict(zip(("out", "ind", "cnt"), b.spherical_avg_voxelize_forward(feat, nc, r))))
    assert scaled_err(A(out), oracle.scatter_mean(A(feat), A(ind), A(cnt), r)) <= TOL
    oi, oc = oracle.sph_grid_stats(A(nc), r)
    mism = int((oi != A(ind)).sum())
    assert mism <= max(2, B * N // 2000), "CPU oracle (libm acosf/atanf) disagrees on %d points" % mism
    if mism == 0:
        omean = oracle.scatter_mean(A(feat), oi, oc, r)
        assert scaled_err(A(out), omean) <= TOL
        if r % 2 == 0:
            assert np.array_equal(A(out), omean)      # tiled and scan-sized paths sum in point order, exactly like the oracle


@pytest.mark.parametrize("B,N,C,r", [(32, 1024, 71, 32), (3, 1000, 5, 16), (2, 2048, 3, 32), (2, 1500, 4, 32), (5, 257, 2, 8),
                                      (1, 64, 150, 32), (2, 300, 3, 2), (2, 1024, 3, 64), (3, 1024, 7, 22)])
def test_cube_devox_streaming_vs_gather_vs_oracle(ri, oracle, B, N, C, r):
    """The three forms of the cube devoxelizer (per-thread global gathers; TMA-streamed planes + shared-memory gathers; the
    default — the cloud's touched 32-byte sectors compacted into shared memory, where it applies) and the C oracle agree bit for bit on outs / inds / wgts — including points on cell boundaries, on the far faces (x = r-1: no
    high corner) and at the grid's corners."""
    import os
    g = torch.Generator().manual_seed(100 + r + N)
    nc = torch.rand(B, 3, N, generator=g) * (r - 1)
    nc[:, :, :N // 8] = torch.round(nc[:, :, :N // 8])                  # integer coordinates: zero high weights
    nc[:, 0, N // 8:N // 6] = r - 1                                     # far x face
    nc[:, :, N // 6:N // 5] = torch.randint(0, 2, (B, 3, N // 5 - N // 6), generator=g).float() * (r - 1)   # corners
    nc = nc.cuda().contiguous()
    grid = torch.randn(B, C, r, r, r, generator=g).cuda()
    res = {}
    L = ri._lib.lib
    try:
        for mode in ("0", "1", "sectors"):
            assert L.ri_debug_set_knob(b"RI_DEVOX_STREAM", -1 if mode == "sectors" else int(mode)) == 0
            res[mode] = torch.ops.ri.trilinear_devox(nc, grid, r)
            torch.cuda.synchronize()
    finally:
        L.ri_debug_set_knob(b"RI_DEVOX_STREAM", -1)
    oo, oi, ow = oracle.trilinear_devoxelize(A(nc), A(grid), r)
    for mode in ("0", "1", "sectors"):
        o, di, dw = res[mode]
        assert np.array_equal(A(di), oi), "corner indices, form %s" % mode
        assert np.array_equal(A(dw), ow), "corner weights, form %s" % mode
        assert np.array_equal(A(o), oo), "devoxelized features, form %s" % mode


@pytest.mark.parametrize("B,N,C,r", [(32, 1024, 71, 32), (4, 900, 6, 16), (2, 5000, 3, 32)])
def test_cube_pipeline_vs_reference(ri, reference, oracle, B, N, C, r):
    pts = clouds(B, N, 21)
    vox_mod = ri.modules.Voxelization(r, normalize=False)
    feat = randn([B, N, C, r], B, C, N)
    out, ind, nc = vox_mod(feat, T(pts[:, :3].copy()))
    vc = torch.round(nc).to(torch.int32).contiguous()
    reference.equal("cube_pipeline/%d-%d-%d-%d" % (B, N, C, r), {"ind": ind.view(B, N)},
                    lambda b: {"ind": b.avg_voxelize_forward(feat, vc, r)[1].view(B, N)})
    grid = randn([B, N, C, r, 8], B, 8, r, r, r)
    d = ri.functional.trilinear_devoxelize(grid, nc, r, True)
    assert np.array_equal(A(d), oracle.trilinear_devoxelize(A(nc), A(grid), r)[0])
    oout, oind, ocnt = oracle.avg_voxelize(A(feat), A(vc), r)
    assert np.array_equal(A(ind), oind)
    assert scaled_err(A(out.reshape(B, C, -1)), oout) <= TOL
    assert np.array_equal(A(out.reshape(B, C, -1)), oout)      # same terms, same (ascending point) order as the oracle: same bits


def test_voxel_means_elementwise_against_reference_noise(ri, oracle):
    """The reference sums a cell's terms with float atomics: its own output changes from run to run, so the means are compared
    with max|d| / max|ref| (`scaled_err`) elsewhere.  This test states the ELEMENT-WISE relative number too, against the exact
    (fp64) mean of every cell: ours (deterministic, ascending point order, bit-equal to the C oracle) differs from it only by
    fp32 rounding, as any fp32 summation order (the reference's atomics included) does, <= 1e-4 relative on every cell whose
    mean is not a near-cancellation (|mean| >= 1e-3 of the largest)."""
    B, N, C, r = 32, 1024, 67, 32
    pts = clouds(B, N, 5)
    nc = sph_norm(T(pts[:, :3].copy()))
    feat = randn([B, N, C, r, 5], B, C, N)
    out, ind, cnt = torch.ops.ri.sph_voxelize(feat, nc, r)
    f, i, c = A(feat).astype(np.float64), A(ind), A(cnt)
    exact = np.zeros((B, r ** 3, C))
    for b in range(B):
        v = i[b] >= 0
        np.add.at(exact[b], i[b][v], f[b][:, v].T)
    exact = exact.transpose(0, 2, 1) / np.maximum(c, 1)[:, None, :]
    got = A(out).astype(np.float64).reshape(B, C, -1)
    keep = np.abs(exact) >= 1e-3 * np.abs(exact).max()
    ours = float(np.max(np.abs(got[keep] - exact[keep]) / np.abs(exact[keep])))
    rec = {"shape": [B, N, C, r], "elementwise_rel_ours_vs_exact": ours, "cells_compared": int(keep.sum()),
           "scaled_ours_vs_exact": scaled_err(got, exact)}
    assert ours <= 1e-4, rec


def test_sph_devox_and_edge_vs_reference(ri, reference, oracle):
    """Corner indices and weights against the reference kernel's; the devoxelized features against the C oracle on every point
    whose corners it reproduces (libm acosf/atanf may move a point on a cell boundary, and round weights 1 ulp apart)."""
    B, N, C, r = 8, 1024, 64, 32
    pts = clouds(B, N, 31)
    nc = sph_norm(T(pts[:, :3].copy()))
    feat = randn([B, N, C, r], B, C, N)
    avg, ind, cnt = torch.ops.ri.sph_voxelize(feat, nc, r)
    grid = randn([B, N, C, r, 1], B, C, r ** 3)
    o, di, dw = torch.ops.ri.sph_trilinear_devox(nc, grid, ind, r)
    reference.equal("sph_devox", {"inds": di, "wgts": dw},
                    lambda b: dict(zip(("out", "inds", "wgts"), b.spherical_trilinear_devoxelize_forward(r, True, nc, grid, ind))))
    oo, odi, odw = oracle.spherical_trilinear_devoxelize(A(nc), A(grid), A(ind), r)
    assert (odi != A(di)).mean() < 1e-3
    same = (odi == A(di)).all(1)                                         # [B, N]: the oracle finds the same 8 corners
    assert scaled_err(A(o).transpose(0, 2, 1)[same], oo.transpose(0, 2, 1)[same]) <= TOL
    # edge features: reference PVConv block, restated with torch ops (pvconv.py:68-90)
    mask = ind == -1
    it = ind.clone(); it[mask] = 0
    centre = avg.gather(2, it.unsqueeze(1).expand(-1, C, -1).long())
    rel = feat - centre
    rel[mask.unsqueeze(1).expand(-1, C, -1)] = 0
    want = torch.cat((rel, feat), 1)
    got = torch.ops.ri.voxel_edge_gather(avg, feat, ind)
    assert torch.equal(got, want)
    assert np.array_equal(A(got), oracle.voxel_edge_gather(A(avg), A(feat), A(ind)))


# ================================================================================================ modules / engine
def test_pvconv_forward_backward(ri):
    torch.manual_seed(0)
    B, N, C = 2, 512, 16
    pts = T(clouds(B, N, 41)[:, :3].copy())
    for shape in ("spherical", "cube"):
        conv = ri.modules.PVConv(C, 32, 'dgcnn_kernel', shape, 3, 16, with_coeff=True, with_se=True, normalize=False).cuda()
        feat = torch.randn(B, C, N, device="cuda", requires_grad=True)
        out, c = conv((feat, pts))
        assert out.shape == (B, 32, N) and torch.isfinite(out).all()
        out.square().mean().backward()
        assert feat.grad is not None and torch.isfinite(feat.grad).all() and float(feat.grad.abs().sum()) > 0
        keys = set(conv.state_dict().keys())
        assert "coefficient" in keys and "voxel_layers.0.weight" in keys and "point_layers.layers.0.weight" in keys


@pytest.mark.parametrize("B,N,C,k,r", [(8, 1024, 19, 20, 32), (3, 2000, 5, 16, 16), (2, 1024, 4, 20, 64), (2, 600, 3, 8, 8),
                                        (2, 5000, 3, 20, 32), (1, 1024, 9, 20, 22)])
def test_frontend_engine_matches_ops(ri, B, N, C, k, r):
    """The engine (one captured step) against the reference-shaped ops, on the fused-prefix path (N <= 1024), the phase-by-phase
    path (N = 2000), the gather devoxelizer (r = 64), the k-NN hash grid + atomic voxelizer fallback (N = 5000) and an odd grid."""
    pts = clouds(B, N, 51); feats = ri.synth.make_features(B, C, N, 51)
    for shape in ("spherical", "cube"):
        fe = ri.FrontEnd(B, N, C, k=k, r=r, voxel_shape=shape)
        res = fe(pts, feats)
        res = {kk: v.clone() for kk, v in res.items()}
        xyz, nrm = T(pts[:, :3].copy()), T(pts[:, 3:].copy())
        _, idx = torch.ops.ri.knn_one(xyz, xyz, k)
        assert torch.equal(torch.ops.ri.ppf_gather(xyz, nrm, idx).cpu(), res["ppf"])
        f = T(feats)
        if shape == "spherical":
            avg, ind, nc = ri.modules.Spherical_Voxelization(r)(f, xyz)
            dv = ri.functional.spherical_trilinear_devoxelize(avg, nc, ind, r)
        else:
            avg, ind, nc = ri.modules.Voxelization(r, normalize=False)(f, xyz)
            dv = ri.functional.trilinear_devoxelize(avg, nc, r)
        edge = ri.functional.voxel_edge_features(avg, f, ind).cpu()
        if N <= 4096:
            assert torch.equal(dv.cpu(), res["devox"])
            assert torch.equal(edge, res["edge"])
            again = fe(pts, feats)                           # graph replay is deterministic
            assert all(torch.equal(again[kk], res[kk]) for kk in res)
        else:
            # beyond the tiled path the voxelizer sums a cell with float atomics (as the reference does): the order, hence
            # the last bits of the means, changes from run to run
            assert scaled_err(A(dv), A(res["devox"])) <= TOL
            assert scaled_err(A(edge), A(res["edge"])) <= TOL


def test_error_behaviour(ri):
    x = torch.randn(2, 3, 64)
    with pytest.raises(RuntimeError):
        torch.ops.ri.knn(x, x, 4)                        # CPU tensor -> RuntimeError, like CHECK_CUDA
    xc = torch.randn(2, 64, 3, device="cuda").transpose(1, 2)
    with pytest.raises(RuntimeError):
        torch.ops.ri.knn(xc, xc, 4)                      # non-contiguous, like CHECK_CONTIGUOUS
    with pytest.raises(RuntimeError):
        torch.ops.ri.cube_voxelize(torch.randn(1, 2, 8, device="cuda"), torch.zeros(1, 3, 8, device="cuda"), 4)  # float coords


# ================================================================================================ fused forms
@pytest.mark.parametrize("shape", ["spherical", "cube"])
def test_voxelize_edge_fused_equals_two_step(ri, shape):
    B, N, C, r = 6, 1024, 13, 32
    pts = clouds(B, N, 61)
    xyz = T(pts[:, :3].copy())
    feat = torch.randn(B, C, N, device="cuda")
    if shape == "spherical":
        nc = sph_norm(xyz); nc[0, :, 7] = 0.0; nc[1, :, 9] = torch.tensor([0.0, 0.0, -0.3], device="cuda")   # undefined pts
        out, ind, cnt = torch.ops.ri.sph_voxelize(feat, nc, r)
        out2, ind2, cnt2, edge = torch.ops.ri.sph_voxelize_edge(feat, nc, r)
        assert int((ind == -1).sum()) >= 2
    else:
        vc = torch.randint(0, r, (B, 3, N), device="cuda", dtype=torch.int32)
        out, ind, cnt = torch.ops.ri.cube_voxelize(feat, vc, r)
        out2, ind2, cnt2, edge = torch.ops.ri.cube_voxelize_edge(feat, vc, r)
    assert torch.equal(out, out2) and torch.equal(ind, ind2) and torch.equal(cnt, cnt2)
    assert torch.equal(edge, torch.ops.ri.voxel_edge_gather(out, feat, ind))


def test_voxelize_many_points_per_tile(ri, oracle):
    """All points inside one grid tile (more occupied cells per tile than the register cache holds) and heavy
    multiplicity per cell."""
    B, N, C, r = 2, 4096, 5, 32
    vc = torch.zeros((B, 3, N), device="cuda", dtype=torch.int32)
    vc[:, 0] = torch.randint(0, 2, (B, N), device="cuda")            # x in {0,1}: cells 0..2047, one tile
    vc[:, 1] = torch.randint(0, 32, (B, N), device="cuda")
    vc[:, 2] = torch.randint(0, 32, (B, N), device="cuda")
    feat = torch.randn(B, C, N, device="cuda")
    out, ind, cnt, edge = torch.ops.ri.cube_voxelize_edge(feat, vc, r)
    oout, oind, ocnt = oracle.avg_voxelize(A(feat), A(vc), r)
    assert np.array_equal(A(ind), oind) and np.array_equal(A(cnt), ocnt)
    assert np.array_equal(A(out), oout)
    assert np.array_equal(A(edge), oracle.voxel_edge_gather(oout, A(feat), oind))


def test_prologue_bit_identical_to_torch(ri):
    """The one-kernel coordinate prologue must reproduce the torch module shells bit for bit (given torch's mean)."""
    L = ri._lib.lib
    B, N, r = 16, 1024, 32
    pts = T(clouds(B, N, 71))
    pts[:, :3] *= 1.7                                               # push some points outside [-1,1] -> clamp path
    xyz = pts[:, :3].contiguous()
    mean = pts[:, :3, :].mean(2)
    assert torch.equal(mean, xyz.mean(2)), "strided-view mean differs from contiguous mean"
    st = torch.cuda.current_stream().cuda_stream
    nc = torch.empty(B, 3, N, device="cuda"); vc = torch.empty(B, 3, N, device="cuda", dtype=torch.int32)
    o_xyz = torch.empty(B, 3, N, device="cuda"); o_n = torch.empty(B, 3, N, device="cuda")
    # cube, normalize=False / True
    for shape, mod in ((0, ri.modules.Voxelization(r, normalize=False)), (1, ri.modules.Voxelization(r, normalize=True, eps=0))):
        t = xyz - xyz.mean(2, keepdim=True)
        if shape == 1:
            t = t / (t.norm(dim=1, keepdim=True).max(dim=2, keepdim=True).values * 2.0 + 0) + 0.5
        else:
            t = (t + 1) / 2.0
        t = torch.clamp(t * r, 0, r - 1)
        ok_modes = []
        for mode in range(5):
            assert L.ri_vox_prologue_f32(pts.data_ptr(), 6, mean.data_ptr(), B, N, r, shape, 0.0, mode, o_xyz.data_ptr(),
                                         o_n.data_ptr(), nc.data_ptr(), vc.data_ptr(), st) == 0
            if torch.equal(nc, t) and torch.equal(vc, torch.round(t).to(torch.int32)):
                ok_modes.append(mode)
        assert ri.FrontEnd.NORM_MODE in ok_modes, "cube shape %d: matching norm modes %s" % (shape, ok_modes)
        assert torch.equal(o_xyz, xyz) and torch.equal(o_n, pts[:, 3:].contiguous())
    # spherical
    t = sph_norm(xyz)
    ok_modes = []
    for mode in range(5):
        assert L.ri_vox_prologue_f32(pts.data_ptr(), 6, mean.data_ptr(), B, N, r, 2, 0.0, mode, None, None,
                                     nc.data_ptr(), None, st) == 0
        if torch.equal(nc, t):
            ok_modes.append(mode)
    assert ri.FrontEnd.NORM_MODE in ok_modes, "spherical: matching norm modes %s" % ok_modes


def test_pvconv_fused_edge_gradients_match_unfused(ri):
    """PVConv uses the fused voxelize+edge op; its gradients must equal the two-step composition's."""
    torch.manual_seed(1)
    B, N, C, r = 2, 256, 6, 8
    xyz = T(clouds(B, N, 81)[:, :3].copy())
    for shape in ("spherical", "cube"):
        mod = ri.modules.Spherical_Voxelization(r) if shape == "spherical" else ri.modules.Voxelization(r, normalize=False)
        f1 = torch.randn(B, C, N, device="cuda", requires_grad=True)
        f2 = f1.detach().clone().requires_grad_(True)
        grid1, ind1, _, edge1 = mod(f1, xyz, with_edge=True)
        grid2, ind2, _ = mod(f2, xyz)
        edge2 = ri.functional.voxel_edge_features(grid2, f2, ind2)
        assert torch.equal(grid1, grid2) and torch.equal(edge1, edge2)
        wg, we = torch.randn_like(grid1), torch.randn_like(edge1)
        ((grid1 * wg).sum() + (edge1 * we).sum()).backward()
        ((grid2 * wg).sum() + (edge2 * we).sum()).backward()
        assert scaled_err(A(f1.grad), A(f2.grad)) <= 1e-5


@pytest.mark.parametrize("shape,normalize", [("spherical", False), ("cube", False), ("cube", True)])
def test_fused_front_equals_separate_phases(ri, shape, normalize):
    """ri_vox_front_f32 (prologue + prepare + means/edge in one launch) + fill == prologue, one-shot voxelize_edge."""
    L = ri._lib
    for B, N, C, r in [(5, 1024, 19, 16), (3, 777, 8, 32), (2, 100, 3, 8)]:
        pts = T(clouds(B, N, 77 + N)); feat = T(np.random.default_rng(N).standard_normal((B, C, N)).astype(np.float32))
        st = torch.cuda.current_stream().cuda_stream
        mean = pts[:, :3, :].mean(2)
        sh = 2 if shape == "spherical" else (1 if normalize else 0)
        s = r ** 3
        def bufs():
            return dict(nc=torch.empty((B, 3, N), device="cuda"), vc=torch.zeros((B, 3, N), dtype=torch.int32, device="cuda"),
                        ind=torch.empty((B, N), dtype=torch.int32, device="cuda"), edge=torch.empty((B, 2 * C, N), device="cuda"),
                        out=torch.empty((B, C, s), device="cuda"), cnt=torch.empty((B, s), dtype=torch.int32, device="cuda"))
        nws = L.lib.ri_voxelize_workspace_bytes(B, C, N, r)
        a, b = bufs(), bufs()
        ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
        L.check(L.lib.ri_vox_front_f32(pts.data_ptr(), 6, mean.data_ptr(), feat.data_ptr(), B, C, N, r, sh, 1e-3, 1,
                                       a["nc"].data_ptr(), a["vc"].data_ptr(), a["ind"].data_ptr(), a["edge"].data_ptr(),
                                       ws.data_ptr(), nws, st), "front")
        L.check(L.lib.ri_voxelize_fill_f32(B, C, N, r, 0, B, a["out"].data_ptr(), a["cnt"].data_ptr(), ws.data_ptr(), nws, st), "fill")
        ws2 = torch.empty(nws, dtype=torch.uint8, device="cuda")
        L.check(L.lib.ri_vox_prologue_f32(pts.data_ptr(), 6, mean.data_ptr(), B, N, r, sh, 1e-3, 1, None, None,
                                          b["nc"].data_ptr(), b["vc"].data_ptr(), st), "prologue")
        if shape == "spherical":
            L.check(L.lib.ri_sph_voxelize_edge_f32(feat.data_ptr(), b["nc"].data_ptr(), B, C, N, r, b["out"].data_ptr(),
                                                   b["ind"].data_ptr(), b["cnt"].data_ptr(), b["edge"].data_ptr(),
                                                   ws2.data_ptr(), nws, st), "vox")
        else:
            L.check(L.lib.ri_cube_voxelize_edge_f32(feat.data_ptr(), b["vc"].data_ptr(), B, C, N, r, b["out"].data_ptr(),
                                                    b["ind"].data_ptr(), b["cnt"].data_ptr(), b["edge"].data_ptr(),
                                                    ws2.data_ptr(), nws, st), "vox")
        for k in a:
            assert torch.equal(a[k], b[k]), (shape, normalize, B, N, C, r, k)


def test_pipeline_matches_single_engine(ri):
    """FrontEndPipeline (overlapped H2D / step / D2H over 3 slots) returns what FrontEnd.__call__ returns, call after call."""
    B, N, C, k, r = 4, 1024, 9, 20, 16
    fe = ri.FrontEnd(B, N, C, k=k, r=r, voxel_shape="cube")
    pipe = ri.FrontEndPipeline(B, N, C, depth=3, k=k, r=r, voxel_shape="cube")
    want = []
    batches = [(clouds(B, N, 100 + q), np.random.default_rng(q).standard_normal((B, C, N)).astype(np.float32)) for q in range(7)]
    for pts, ft in batches:
        out = fe(pts, ft)
        want.append({n: v.clone() for n, v in out.items()})
    tickets = []
    got = [None] * len(batches)
    for q, (pts, ft) in enumerate(batches):
        s = pipe.acquire()
        if len(tickets) >= pipe.depth:                       # the slot being reused: its result was collected below
            pass
        pipe.slot(s).h_points.copy_(torch.from_numpy(pts)); pipe.slot(s).h_features.copy_(torch.from_numpy(ft))
        pipe.submit(s)
        tickets.append((q, s))
        if len(tickets) == pipe.depth:                       # collect the oldest before its slot comes round again
            q0, s0 = tickets.pop(0)
            got[q0] = {n: v.clone() for n, v in pipe.result(s0).items()}
    for q0, s0 in tickets:
        got[q0] = {n: v.clone() for n, v in pipe.result(s0).items()}
    for a, b in zip(want, got):
        for n in a:
            assert torch.equal(a[n], b[n]), n


@pytest.mark.parametrize("shape", ["cube", "spherical"])
def test_lanes_match_serial_engine(ri, shape):
    """FrontEndLanes (three batches in flight on three launch streams) leaves in every engine exactly what a serial replay
    of that engine leaves — concurrency changes no bit."""
    B, N, C, k, r = 8, 1024, 11, 20, 32
    engines, want = [], []
    for q in range(3):
        fe = ri.FrontEnd(B, N, C, k=k, r=r, voxel_shape=shape)
        fe.load(clouds(B, N, 300 + q), np.random.default_rng(q).standard_normal((B, C, N)).astype(np.float32))
        fe.forward(); torch.cuda.synchronize()
        want.append({n: getattr(fe, n).clone() for n in ("ppf", "knn_idx", "grid", "cnt", "ind", "devox", "edge")})
        for n in want[-1]:
            getattr(fe, n).zero_()
        engines.append(fe)
    lanes = ri.FrontEndLanes(engines, lanes=3)
    lanes.begin()
    for i in range(9):
        lanes.forward(i)
    lanes.end()
    torch.cuda.synchronize()
    for fe, w in zip(engines, want):
        for n, v in w.items():
            assert torch.equal(getattr(fe, n), v), n
    # stress: 900 more steps in flight (persistent TMA kernels, mbarrier rings, dynamic work counters) — same bits at the end
    lanes.begin()
    for i in range(900):
        lanes.forward(i)
    lanes.end()
    torch.cuda.synchronize()
    for fe, w in zip(engines, want):
        for n, v in w.items():
            assert torch.equal(getattr(fe, n), v), "after 900 steps: " + n


@pytest.mark.parametrize("k,n,m", [(20, 1024, 1024), (8, 100, 777), (16, 1000, 3000), (32, 333, 64), (20, 5, 3)])
def test_knn_ties_and_short_reference_sets_vs_oracle(ri, oracle, k, n, m):
    """Every reference point duplicated (distance ties everywhere), queries sitting on references (d = 0), fewer references
    than k, reference sets larger than one shared-memory tile: indices and distances equal the oracle's bit for bit."""
    g = torch.Generator().manual_seed(k * 1000 + n)
    x1 = torch.randn(3, 3, n, generator=g)
    x2 = torch.randn(3, 3, m, generator=g)
    x2[:, :, m // 2:] = x2[:, :, :m - m // 2]
    x1[:, :, :min(n, m) // 4] = x2[:, :, :min(n, m) // 4]
    x1, x2 = x1.cuda().contiguous(), x2.cuda().contiguous()
    d1, d2, i1, i2 = torch.ops.ri.knn(x1, x2, k)
    od1, od2, oi1, oi2 = oracle.knn(A(x1), A(x2), k)
    assert np.array_equal(A(i1), oi1) and np.array_equal(A(i2), oi2)
    assert np.array_equal(A(d1), od1) and np.array_equal(A(d2), od2)


@pytest.mark.parametrize("B,N", [(32, 1024), (6, 1000), (8, 128), (16, 512), (1, 1024), (5, 512)])
def test_in_kernel_mean_reproduces_torch(ri, B, N):
    """The fused prefix kernel's own per-cloud mean (torch's reduction order restated, csrc/voxelize.cu) equals
    `coords.mean(2)` bit for bit on awkward data, and the engine only drops the torch kernel after checking that itself."""
    fe = ri.FrontEnd(B, N, 5, k=8, r=16, voxel_shape="cube")
    g = torch.Generator(device="cuda"); g.manual_seed(N)
    pts = torch.randn((B, 6, N), device="cuda", generator=g) * 5 - 1.3
    pts[:, :3, ::5] *= 300.0
    fe.load(pts, torch.randn((B, 5, N), device="cuda", generator=g))
    fe.forward(); torch.cuda.synchronize()
    assert fe._own_mean_checked
    if 3 * B >= 16:
        assert fe._own_mean, "the engine did not accept the in-kernel mean for this shape"
        assert torch.equal(fe._mean_buf, pts[:, :3, :].mean(2))
    else:
        assert not fe._own_mean                            # few outputs: torch reduces with wider blocks, the engine keeps torch's kernel
    # and the step built on it still equals the module path (torch mean) bit for bit
    vox = ri.modules.Voxelization(16, normalize=False)
    avg, ind, nc = vox(fe.features, pts[:, :3].contiguous())
    assert torch.equal(ind, fe.ind) and torch.equal(nc, fe.norm_coords) and torch.equal(avg.reshape(B, 5, -1), fe.grid.reshape(B, 5, -1))
