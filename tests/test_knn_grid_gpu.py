"""GPU parity of the hash-grid k-NN (csrc/knn_grid.cu) — results must be BIT-IDENTICAL to the brute-force search:
against ri_knn_f32 (itself pinned to the reference's KnnKernel and the golden vectors in test_parity_gpu.py), against
what the reference's own kernel returns on one scan-sized cloud, and against the C oracle on small cases.  Covers the edge cases
of knn/knn.cu:5-49: distance ties (duplicated points -> lower index first), m < k (sentinel slots), queries outside
the reference bounding box, d^2 >= 10000 never inserted, degenerate (flat / single-point) clouds."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ri():
    import ri_b200
    return ri_b200


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def both(x1, x2, k):
    L = __import__("ri_b200")._lib
    q, r = T(x1), T(x2)
    B, _, n = q.shape; m = r.shape[2]
    d0 = torch.empty((B, k, n), device="cuda"); i0 = torch.empty((B, k, n), dtype=torch.int32, device="cuda")
    L.check(L.lib.ri_knn_f32(q.data_ptr(), r.data_ptr(), B, 3, n, m, k, d0.data_ptr(), i0.data_ptr(),
                             torch.cuda.current_stream().cuda_stream), "brute")
    d1, i1 = torch.ops.ri.knn_grid(q, r, k)
    return d0, i0, d1, i1


@pytest.mark.parametrize("n,m,k", [(1024, 1024, 20), (5000, 5000, 20), (333, 7001, 16), (2000, 50, 8), (100, 10, 20),
                                    (777, 4096, 32), (64, 1, 4)])
def test_grid_equals_brute_force_on_clouds(ri, oracle, n, m, k):
    from ri_b200 import synth
    B = 3
    x1 = synth.make_clouds(B, n, seed=5)[:, :3].copy(); x2 = synth.make_clouds(B, m, seed=6)[:, :3].copy()
    q = min(n, m) // 2
    x2[:, :, :q] = x1[:, :, :q]                                       # shared points: d = 0
    if m >= 8:
        x2[:, :, m - 4:] = x2[:, :, :4]                               # exact duplicates -> index tie-break
    d0, i0, d1, i1 = both(x1, x2, k)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    if n * m <= 1024 * 1024:
        od, oi = oracle.knn_one(x1, x2, k)
        assert np.array_equal(i1.cpu().numpy(), oi) and np.array_equal(d1.cpu().numpy(), od)


def test_grid_on_scan_sized_cloud_vs_reference_kernel(ri, reference):
    """BASELINE configs[3]: ICL-NUIM-shaped scan, ~50k points, k = 20, self query."""
    from ri_b200 import synth
    x = np.stack([synth.make_scan(50000, seed=s)[:3] for s in range(2)])
    d0, i0, d1, i1 = both(x, x, 20)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    assert bool((d1[:, 0] == 0).all()) and bool((d1[:, 1:] >= d1[:, :-1]).all())
    reference.equal("knn_grid_scan", {"idx": i1[:1], "dist": d1[:1]},  # the reference's own O(n m k) kernel on one scan
                    lambda b: dict(zip(("dist", "_", "idx", "__"), b.knn_forward_cuda(T(x[:1]), T(x[:1]), 20))))
    # the size-routed public op takes the grid path at this size and returns the same thing
    d2, i2 = torch.ops.ri.knn_one(T(x), T(x), 20)
    assert torch.equal(i2, i1) and torch.equal(d2, d1)


def test_grid_edge_cases(ri):
    g = np.random.default_rng(0)
    # heavy ties: points on an integer lattice (many exactly equal distances)
    lat = np.stack(np.meshgrid(np.arange(12), np.arange(12), np.arange(12), indexing="ij")).reshape(3, -1)
    lat = lat[:, g.permutation(lat.shape[1])].astype(np.float32)[None]
    d0, i0, d1, i1 = both(lat, lat, 20)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    # flat cloud (zero extent on one axis) and a single repeated point
    flat = g.standard_normal((2, 3, 3000)).astype(np.float32); flat[:, 2] = 0.25
    d0, i0, d1, i1 = both(flat, flat, 16)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    same = np.ones((1, 3, 500), np.float32)
    d0, i0, d1, i1 = both(same, same, 8)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    assert np.array_equal(i1[0, :, 0].cpu().numpy(), np.arange(8))    # all distances 0: indices ascending
    # queries far outside the references' box, some farther than sqrt(10000): those never enter
    refs = g.uniform(-1, 1, (2, 3, 2500)).astype(np.float32)
    qs = g.uniform(-1, 1, (2, 3, 600)).astype(np.float32)
    qs[:, :, :100] += 50.0; qs[:, :, 100:200] -= 90.0; qs[:, 0, 200:300] += 3.0
    d0, i0, d1, i1 = both(qs, refs, 20)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    assert bool((d1[:, :, 100:200] == 10000.0).all()) and bool((i1[:, :, 100:200] == 0).all())
    # clustered data: two tight blobs far apart (most cells empty, rings must expand)
    blob = np.concatenate([g.normal(0, 0.01, (1, 3, 1500)), g.normal(5, 0.01, (1, 3, 7))], 2).astype(np.float32)
    d0, i0, d1, i1 = both(blob, blob, 20)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)


def test_grid_errors(ri):
    x = torch.randn(1, 4, 100, device="cuda")
    with pytest.raises(RuntimeError):
        torch.ops.ri.knn_grid(x, x, 8)
    L = ri._lib
    assert L.lib.ri_knn_grid_f32(0, 0, 1, 10, 10, 64, 0, 0, 0, 0, 0) == -3      # k > 32 unsupported
    assert L.lib.ri_knn_grid_f32(0, 0, 1, 10, 10, 8, 0, 0, 0, 0, 0) == -2       # workspace missing
