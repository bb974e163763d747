"""Row f12 (SURVEY.md §8f): the vectorised farthest point sampling oracle (tests/fps_oracle.py) against the contract's
literal per-point loop, and the properties the contract implies.  CPU only."""
import numpy as np
import pytest

import fps_oracle as ref


def _cases():
    for name, make in ref.HAND_MADE.items():
        yield name, make()
    rng = np.random.default_rng(5)
    yield "random", rng.standard_normal((3, 40)).astype(np.float32)


@pytest.mark.parametrize("name,xyz", list(_cases()), ids=[c[0] for c in _cases()])
def test_oracle_equals_literal_loop(name, xyz):
    N = xyz.shape[1]
    for n in sorted({0, 1, 2, N // 2, N - 1, N}):
        for m in sorted({1, 2, max(n - 1, 1), max(n, 1), n + 3}):
            assert ref.fps_one(xyz, n, m).tolist() == ref.fps_literal(xyz, n, m), (name, n, m)


def test_empty_cloud_gives_minus_one():
    assert ref.fps_one(np.zeros((3, 5), np.float32), 0, 4).tolist() == [-1] * 4


def test_single_point_repeats():
    assert ref.fps_one(np.ones((3, 5), np.float32), 1, 3).tolist() == [0, 0, 0]


def test_m_above_n_repeats_the_last_pick():
    xyz = ref.collinear(6)
    idx = ref.fps_one(xyz, 6, 10).tolist()
    assert sorted(idx[:6]) == list(range(6)) and idx[6:] == [idx[5]] * 4


def test_collinear_alternates_ends():
    assert ref.fps_one(ref.collinear(17), 17, 3).tolist() == [0, 16, 8]


def test_lattice_ties_take_the_lowest_index():
    xyz = ref.lattice(4)
    idx = ref.fps_one(xyz, xyz.shape[1], 2).tolist()
    assert idx == [0, xyz.shape[1] - 1]            # (3,3,3) is the unique farthest corner
    idx = ref.fps_one(xyz, xyz.shape[1], 64).tolist()
    assert sorted(idx) == list(range(64))           # every lattice point once: there are no duplicates


def test_duplicates_are_never_taken():
    xyz = ref.duplicates()
    idx = ref.fps_one(xyz, xyz.shape[1], xyz.shape[1]).tolist()
    distinct = {tuple(xyz[:, i]) for i in range(xyz.shape[1])}
    picked = [tuple(xyz[:, i]) for i in idx]
    first = picked[:len(distinct)]
    assert len(set(first)) == len(distinct)
    assert idx[len(distinct):] == [idx[len(distinct) - 1]] * (len(idx) - len(distinct))


def test_identical_points_repeat_index_zero():
    assert ref.fps_one(ref.identical(), 9, 5).tolist() == [0] * 5


def test_nan_point_is_taken_then_repeats():
    xyz = ref.with_nan(at=7)
    idx = ref.fps_one(xyz, 20, 6).tolist()
    assert idx[0] == 0 and idx[1] == 7 and idx[2:] == [7] * 4


def test_padding_is_not_read():
    rng = np.random.default_rng(3)
    xyz = rng.standard_normal((3, 30)).astype(np.float32)
    pad = xyz.copy()
    pad[:, 20:] = np.nan
    assert ref.fps_one(xyz, 20, 25).tolist() == ref.fps_one(pad, 20, 25).tolist()
