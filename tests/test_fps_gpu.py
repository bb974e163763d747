"""Row f12 (SURVEY.md §8f): batched farthest point sampling on the GPU (csrc/fps.cu) against the fp64 replay of its
contract (tests/fps_oracle.py), bit for bit, on every cluster size the launch picks."""
import numpy as np
import pytest

import fps_oracle as ref

pytestmark = pytest.mark.gpu


def _fps(xyz, m, lengths=None):
    import torch
    import ri_b200  # noqa: F401
    t = torch.from_numpy(np.ascontiguousarray(xyz, np.float32)).cuda()
    lens = None if lengths is None else torch.tensor(list(lengths), dtype=torch.int32)
    return torch.ops.ri.furthest_point_sample(t, lens, int(m)).cpu().numpy()


def _check(xyz, m, lengths=None):
    got = _fps(xyz, m, lengths)
    want = ref.fps(xyz, m, lengths)
    assert got.dtype == np.int32 and got.shape == want.shape
    bad = np.nonzero((got != want).any(1))[0]
    assert bad.size == 0, "clouds %s differ; first: got %s want %s" % (bad[:5], got[bad[0]][:16], want[bad[0]][:16])
    return got


def _scan_clouds(B, raw, cell, seed):
    import torch
    import ri_b200
    clouds = [torch.from_numpy(np.ascontiguousarray(ri_b200.synth.make_scan(raw, seed=seed + b).T)).cuda() for b in range(B)]
    return ri_b200.grid_sub_sampling_many([(c[:, :3].contiguous(), c[:, 3:].contiguous()) for c in clouds], grid_size=cell)


def test_modelnet_clouds():
    import ri_b200
    c = ri_b200.synth.make_clouds(64, 1024, seed=12)
    _check(np.ascontiguousarray(c[:, :3]), 512)


# N just below and above every switch of the launch: threads per CTA (32 .. 512 with 16 points each), the cluster size
# (doubled from 1 while each CTA keeps >= 1024 points; the fewest CTAs of <= 8192 points), 16-CTA clusters above 65536.
SWITCH_N = [1, 2, 511, 512, 513, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4096, 4097, 8191, 8192, 8193, 16384, 16385,
            32768, 32769, 65536, 65537, 131072]


@pytest.mark.parametrize("N", SWITCH_N)
@pytest.mark.parametrize("B", [1, 3])
def test_sizes_around_every_switch(N, B):
    rng = np.random.default_rng(N + B)
    xyz = rng.uniform(-1, 1, (B, 3, N)).astype(np.float32)
    _check(xyz, min(N + 2, 48))


@pytest.mark.parametrize("N", [8192, 8193])
def test_wide_batch_cluster_sizes(N):
    rng = np.random.default_rng(N)
    xyz = rng.standard_normal((64, 3, N)).astype(np.float32)
    _check(xyz, 24)


def test_ragged_batch_with_poisoned_padding():
    m, N = 40, 3000
    ns = [0, 1, 2, m - 1, m, m + 1, 1000, 2047, N]
    rng = np.random.default_rng(7)
    xyz = rng.uniform(-2, 2, (len(ns), 3, N)).astype(np.float32)
    for b, n in enumerate(ns):
        xyz[b, :, n:] = np.nan if b % 2 else 1e30
    got = _check(xyz, m, ns)
    assert (got[0] == -1).all() and (got[1] == 0).all()


@pytest.mark.parametrize("name", sorted(ref.HAND_MADE))
def test_hand_made_clouds(name):
    xyz = ref.HAND_MADE[name]()
    n = xyz.shape[1]
    for m in (1, n, n + 5):
        _check(xyz[None], m)


def test_scans():
    subs = _scan_clouds(2, 200000, 0.03, seed=40)
    for p, _, _ in subs:
        xyz = p.t().contiguous().cpu().numpy()[None]
        assert 30000 < xyz.shape[2] <= 131072
        _check(xyz, 2048)


def test_batch_independence_and_determinism():
    rng = np.random.default_rng(9)
    N, ns = 20000, [20000, 5000, 17, 12000]
    xyz = rng.standard_normal((4, 3, N)).astype(np.float32)
    a = _fps(xyz, 300, ns)
    assert np.array_equal(a, _fps(xyz, 300, ns))
    for b, n in enumerate(ns):
        assert np.array_equal(a[b], _fps(xyz[b:b + 1, :, :n], 300)[0])


def test_gather_features_match_torch():
    import torch
    from ri_b200 import _backend
    from ri_b200.functional import gather
    g = torch.Generator().manual_seed(3)
    feats = torch.randn(3, 5, 100, generator=g).cuda()
    idx = torch.randint(0, 100, (3, 40), generator=g, dtype=torch.int32).cuda()
    idx[:, 1] = idx[:, 0]                                      # repeated indices: the backward sums them
    want = torch.gather(feats, 2, idx.long().unsqueeze(1).expand(3, 5, 40))
    assert torch.equal(_backend.gather_features_forward(feats, idx), want)
    gy = torch.randn(3, 5, 40, generator=g).cuda()
    gw = torch.zeros(3, 5, 100, device="cuda")
    for b in range(3):
        gw[b].index_add_(1, idx[b].long(), gy[b])
    gb = _backend.gather_features_backward(gy, idx, 100)
    assert torch.allclose(gb, gw, rtol=0, atol=1e-6)
    x = feats.clone().requires_grad_(True)
    gather(x, idx).backward(gy)
    assert torch.allclose(x.grad, gw, rtol=0, atol=1e-6)


def test_functional_and_backend():
    import torch
    import ri_b200
    from ri_b200.functional import furthest_point_sample
    c = ri_b200.synth.make_clouds(4, 1024, seed=5)
    xyz = torch.from_numpy(np.ascontiguousarray(c[:, :3])).cuda()
    want = ref.fps(c[:, :3], 128)
    out, idx = furthest_point_sample(xyz, 128, return_indices=True)
    assert np.array_equal(idx.cpu().numpy(), want)
    assert torch.equal(out, torch.gather(xyz, 2, idx.long().unsqueeze(1).expand(4, 3, 128)))
    assert torch.equal(furthest_point_sample(xyz, 128), out)
    assert np.array_equal(ri_b200._backend.furthest_point_sampling(xyz, 128).cpu().numpy(), want)
    out, idx = furthest_point_sample(xyz, 16, lengths=[1024, 0, 3, 700], return_indices=True)
    assert np.array_equal(idx.cpu().numpy(), ref.fps(c[:, :3], 16, [1024, 0, 3, 700]))


def test_farthest_point_batch_on_grid_subsampled_scans():
    import torch
    import ri_b200
    subs = _scan_clouds(3, 120000, 0.05, seed=70)
    m = 1024
    pts, feats, idx = ri_b200.farthest_point_batch(subs, m)
    assert pts.shape == (3, m, 3) and feats.shape == (3, m, 3) and idx.shape == (3, m)
    for b, (p, f, _) in enumerate(subs):
        want = ref.fps_one(p.t().contiguous().cpu().numpy(), p.shape[0], m)
        assert np.array_equal(idx[b].cpu().numpy(), want)
        assert torch.equal(pts[b], p[idx[b].long()]) and torch.equal(feats[b], f[idx[b].long()])
    pts2, none, idx2 = ri_b200.farthest_point_batch([p for p, _, _ in subs], m)
    assert none is None and torch.equal(idx2, idx) and torch.equal(pts2, pts)


def test_argument_errors_before_launch():
    import torch
    import ri_b200  # noqa: F401
    op = torch.ops.ri.furthest_point_sample
    x = torch.zeros(2, 3, 10, device="cuda")
    cases = [
        (x.double(), None, 4), (x.cpu(), None, 4), (x[:, :2].contiguous(), None, 4), (x.transpose(1, 2), None, 4),
        (x, None, 0), (x, torch.tensor([10, 11], dtype=torch.int32), 4), (x, torch.tensor([-1, 3], dtype=torch.int32), 4),
        (x, torch.tensor([10], dtype=torch.int32), 4), (x, torch.tensor([10, 10]), 4),
        (x, torch.tensor([10, 10], dtype=torch.int32, device="cuda"), 4),
        (torch.zeros(1, 3, 131073, device="cuda"), None, 4),
    ]
    for xyz, lens, m in cases:
        with pytest.raises(RuntimeError):
            op(xyz, lens, m)
    torch.cuda.synchronize()
