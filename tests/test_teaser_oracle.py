"""CPU self-test of tests/teaser_oracle.py (row f10): the clique search against networkx, its tie rule and budget, GNC-TLS
and adaptive voting against ground truth and brute force, and the degenerate cases."""
import networkx as nx
import numpy as np
import pytest

import pose_oracle as po
import teaser_oracle as to


def random_rows(rng, n, p, plant=0):
    """Rows of G(n, p) with a planted clique of `plant` random vertices -> (rows, networkx graph)."""
    A = np.triu(rng.random((n, n)) < p, 1)
    if plant:
        S = rng.choice(n, plant, replace=False)
        A[np.ix_(S, S)] = True
    A = np.triu(A, 1)
    A = A | A.T
    return to.bit_rows(A), nx.from_numpy_array(A.astype(np.uint8))


def is_clique(rows, C):
    return all(rows[u] >> v & 1 for u in C for v in C if u != v)


@pytest.mark.parametrize("n,p,plant,seed", [(40, 0.3, 0, 0), (60, 0.5, 0, 1), (80, 0.2, 12, 2), (120, 0.1, 20, 3),
                                            (50, 0.8, 0, 4), (200, 0.05, 30, 5)])
def test_clique_is_maximum(n, p, plant, seed):
    rows, G = random_rows(np.random.default_rng(seed), n, p, plant)
    c = to.max_clique(rows, 1 << 30)
    assert c.exact and is_clique(rows, c.ranks)
    assert len(c.ranks) == max(len(q) for q in nx.find_cliques(G))


@pytest.mark.parametrize("outliers,seed", [(0.5, 0), (0.9, 1)])
def test_clique_of_matches_is_maximum(outliers, seed):
    a, b, _, _ = po.planted_matches(np.random.default_rng(seed), 150, outliers)
    clique, c = to.clique_of(a, b, 0.03)
    G = nx.from_numpy_array(to.adjacency(a, b, to.beta_of(0.03, 1.0)).astype(np.uint8))
    assert c.exact and np.all(np.diff(clique) > 0)
    assert len(clique) == max(len(q) for q in nx.find_cliques(G))
    assert all(G.has_edge(int(u), int(v)) for u in clique for v in clique if u != v)


def test_tie_rule():
    # two disjoint triangles {0, 2, 4} and {1, 3, 5} (ranks): the greedy start from rank 0 finds the first, the exact search
    # finds nothing strictly larger, so the first one found is kept
    A = np.zeros((6, 6), bool)
    for tri in ((0, 2, 4), (1, 3, 5)):
        for u in tri:
            for v in tri:
                A[u, v] = u != v
    c = to.max_clique(to.bit_rows(A), 100)
    assert c.ranks == [0, 2, 4] and c.exact


def test_budget_exhaustion():
    rows, G = random_rows(np.random.default_rng(11), 90, 0.6)
    full = to.max_clique(rows, 1 << 30)
    assert full.exact and full.nodes > 3
    for budget in (1, 2, full.nodes - 1):
        c = to.max_clique(rows, budget)
        assert not c.exact and c.nodes == budget
        assert is_clique(rows, c.ranks) and c.heuristic <= len(c.ranks) <= len(full.ranks)
    c = to.max_clique(rows, full.nodes)
    assert c.exact and c.ranks == full.ranks


def rot_err_deg(R, gt):
    return np.degrees(np.arccos(np.clip((np.trace(R @ gt[:3, :3].T) - 1) / 2, -1, 1)))


@pytest.mark.parametrize("outliers", [0.5, 0.9, 0.95])
def test_recovers_ground_truth(outliers):
    rng = np.random.default_rng(int(outliers * 100))
    a, b, gt, bad = po.planted_matches(rng, 400, outliers)
    r = to.replay(a, b, 0.03)
    assert r.posed and r.search.exact
    assert rot_err_deg(r.T[:3, :3], gt) < 1.0
    assert np.linalg.norm(r.T[:3, 3] - gt[:3, 3]) < 0.02
    assert r.inliers >= 0.8 * (~bad).sum()


def test_gnc_tls_rejects_outlier_tims():
    # GNC-TLS alone (no clique pruning) over TIMs with 50 % outliers
    rng = np.random.default_rng(3)
    gt = po.rand_pose(rng)
    v = rng.uniform(-1, 1, (200, 3))
    w = v @ gt[:3, :3].T + rng.normal(0, 0.002, v.shape)
    w[:100] = rng.uniform(-1, 1, (100, 3))
    g = to.gnc_tls(v, w, 0.02 ** 2)
    assert rot_err_deg(g.R, gt) < 0.5


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_voting_is_tls_minimum(seed):
    rng = np.random.default_rng(seed)
    x = np.concatenate([rng.normal(0.3, 0.01, 40), rng.uniform(-2, 2, 60)])
    r = 0.03
    est, cost, inside = to.adaptive_voting(x, r)
    grid = np.linspace(x.min() - r, x.max() + r, 200001)
    brute = min(to.tls_cost(x, r, t) for t in grid[::50])
    fine = grid[np.argmin([to.tls_cost(x, r, t) for t in grid])]
    assert to.tls_cost(x, r, est) <= to.tls_cost(x, r, fine) + 1e-9
    assert to.tls_cost(x, r, est) <= brute + 1e-9
    assert abs(est - fine) < 1e-3
    assert cost >= to.tls_cost(x, r, est) - 1e-12         # the voting cost bounds the TLS cost at its estimate


def test_noise_free_is_kabsch():
    rng = np.random.default_rng(7)
    a, b, gt, _ = po.planted_matches(rng, 100, 0.0, noise=0.0)
    r = to.replay(a, b, 0.01)
    assert len(r.clique) == 100 and r.search.exact
    assert np.abs(r.T[:3, :3] - gt[:3, :3]).max() < 1e-6
    assert np.abs(r.T[:3, 3] - gt[:3, 3]).max() < 1e-6


def test_degenerate_give_identity():
    rng = np.random.default_rng(8)
    a, b, _, _ = po.planted_matches(rng, 10, 1.0)
    for m in (0, 1, 2):
        r = to.replay(a[:m], b[:m], 0.01)
        assert not r.posed and np.array_equal(r.T32, np.eye(4, dtype=np.float32)) and r.inliers == 0
    # three matches whose lengths all disagree: the clique has fewer than 3 vertices
    a3 = np.array([[0, 0, 0], [1, 0, 0], [0, 2, 0]], np.float32)
    b3 = np.array([[0, 0, 0], [3, 0, 0], [0, 7, 0]], np.float32)
    r = to.replay(a3, b3, 0.01)
    assert len(r.clique) < 3 and not r.posed and r.inliers == 0
