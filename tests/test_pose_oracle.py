"""CPU self-test of the pose replay (tests/pose_oracle.py, row f3): the sampler's contract, the hypothesis of an exact
triple, recovery of a planted pose, and the ambiguity flags.  No GPU needed."""
import numpy as np
import pytest

import pose_oracle as ref


def test_mix64_known_values():
    # splitmix64 of the state after one increment: mix64(0) is the first output of splitmix64 seeded with 0
    assert ref.mix64(0) == 0xE220A8397B1DCDAF
    assert ref.mix64(1) == ref.mix64(np.array([1], np.uint64))[0]
    x = np.array([0, 1, 2 ** 63 + 5, 2 ** 64 - 1], np.uint64)
    assert [int(v) for v in ref.mix64(x)] == [ref.mix64(int(v)) for v in x]


def test_sample3_distinct_and_in_range():
    hyps = np.arange(64)
    for M in list(range(3, 200)) + [1023, 1024, 4095, 4096, 4097, 5000]:
        for seed, pair in ((0, 0), (2 ** 63 + 5, 3), (12345, 65534)):
            s = ref.sample3(seed, pair, hyps, M)
            assert s.min() >= 0 and s.max() < M, M
            assert np.all((s[:, 0] != s[:, 1]) & (s[:, 1] != s[:, 2]) & (s[:, 0] != s[:, 2])), M


def test_sample3_m3_is_a_permutation():
    s = ref.sample3(7, 1, np.arange(500), 3)
    assert np.all(np.sort(s, 1) == [0, 1, 2])
    assert len({tuple(r) for r in s}) == 6                          # every ordering occurs


def test_sample3_scalar_matches_vector_and_uses_all_seed_bits():
    for h in (0, 1, 127, 128, 999):
        assert ref.sample3(2 ** 63 + 5, 2, h, 4097) == tuple(ref.sample3(2 ** 63 + 5, 2, np.array([h]), 4097)[0])
    a = ref.sample3(5, 0, np.arange(256), 1 << 20)
    b = ref.sample3(2 ** 63 + 5, 0, np.arange(256), 1 << 20)
    assert not np.array_equal(a, b)                                 # the top bit of the seed changes the samples
    assert not np.array_equal(ref.sample3(5, 0, np.arange(256), 1 << 20), ref.sample3(5, 1, np.arange(256), 1 << 20))


def test_hypothesis_of_exact_triples_reproduces_pose():
    rng = np.random.default_rng(0)
    a, b, gt, _ = ref.planted_matches(rng, 50, 0.0, noise=0.0)
    a, b = a.astype(np.float64), a.astype(np.float64) @ gt[:3, :3].T + gt[:3, 3]
    hy = ref.hypotheses(a, b, 40, seed=3, pair=0, thresh=0.01, edge_sim=0.99)
    assert hy.valid.all() and not hy.amb.any()
    assert np.abs(hy.T - gt).max() < 1e-12


def test_replay_recovers_planted_pose_under_70_percent_outliers():
    rng = np.random.default_rng(1)
    a, b, gt, bad = ref.planted_matches(rng, 1500, 0.7)
    r = ref.replay(a, b, hyps=1000, thresh=0.08, seed=1)
    assert r.unambiguous and r.winner >= 0
    assert np.abs(r.T - gt).max() < 5e-3
    assert r.inliers >= 0.95 * (~bad).sum()
    assert r.best_key >> 32 == ref.count_interval(ref.hypotheses(a, b, 1000, 1, 0, 0.08, 0.9).T[r.winner], a, b, 0.08, 0, 0)[0]
    assert (r.best_key & 0xFFFFFFFF) == 0xFFFFFFFF - r.winner
    # Kabsch mode is the SVD fit over every match
    k = ref.replay(a[~bad], b[~bad], hyps=0, thresh=0.08)
    assert np.abs(k.T - gt).max() < 5e-3 and k.inliers == (~bad).sum()


def test_replay_degenerate():
    assert ref.replay(np.zeros((2, 3)), np.zeros((2, 3)), 100, 0.1).T.tolist() == np.eye(4).tolist()
    line = np.zeros((40, 3)); line[:, 0] = np.arange(40) * 0.125
    r = ref.replay(line, line, 500, 0.1)
    assert r.winner == -1 and r.inliers == 0 and np.array_equal(r.T, np.eye(4))
    # fp32 rounding of a coordinate exceeds the 1e-6 norm guard, so the replay cannot promise the GPU agrees
    assert not r.unambiguous


def test_flags_fire_on_the_threshold():
    T = np.eye(4)
    a = np.zeros((3, 3)); b = np.array([[0.08, 0, 0], [0.05, 0, 0], [0.2, 0, 0]])
    assert ref.count_interval(T, a, b, 0.08, 1e-6) == (1, 2)         # the residual on the threshold is "maybe"
    assert ref.count_interval(T, a, b, 0.08, 0.0, 0.0)[0] == 1       # zero band: lo is the strict fp64 count
    # a sample whose own residual sits on the threshold: ambiguous, whichever way fp64 decides it
    rng = np.random.default_rng(2)
    a3 = rng.uniform(-1, 1, (3, 3)); b3 = a3 + rng.normal(0, 0.01, (3, 3))
    hy = ref.hypotheses(a3, b3, 6, 0, 0, thresh=1.0, edge_sim=0.9)
    assert hy.valid.all() and not hy.amb.any()
    A, B = a3[hy.idx[0]], b3[hy.idx[0]]
    d = np.linalg.norm(A @ hy.T[0, :3, :3].T + hy.T[0, :3, 3] - B, axis=1).max()
    for thresh in (d, np.nextafter(d, 1)):
        hy = ref.hypotheses(a3, b3, 6, 0, 0, thresh=thresh, edge_sim=0.9)
        assert hy.amb[0]                                            # the other orderings give other frames
    # an edge ratio exactly at edge_similarity, and a coincident pair of sample points (norm guard), likewise
    assert ref.hypotheses(a3, a3 * 0.5, 6, 0, 0, thresh=10.0, edge_sim=0.5).amb.all()
    a3[1] = a3[0] + [1e-6, 0, 0]
    hy = ref.hypotheses(a3, a3, 60, 0, 0, thresh=10.0, edge_sim=0.9)
    first_edge = np.all(np.sort(hy.idx[:, :2], 1) == [0, 1], 1)
    assert first_edge.any() and np.all(hy.amb[first_edge])           # u = p1 - p0 is the 1e-6 edge


@pytest.mark.parametrize("outliers", [0.3, 0.7])
def test_replay_winner_rule(outliers):
    """The winner has the largest count and the lowest id among equal counts; the key packs both as the kernel does."""
    rng = np.random.default_rng(4)
    a, b, gt, bad = ref.planted_matches(rng, 400, outliers)
    hy = ref.hypotheses(a, b, 300, 9, 2, 0.08, 0.9)
    lo, hi, nom = ref.hypothesis_counts(hy, a, b, 0.08)
    nom = np.where(hy.valid, nom, -1)
    r = ref.replay(a, b, 300, 0.08, seed=9, pair=2)
    assert nom[r.winner] == nom.max() and np.all(nom[:r.winner] < nom.max())
    assert lo[r.winner] <= nom[r.winner] <= hi[r.winner]
