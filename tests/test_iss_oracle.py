"""CPU checks of tests/iss_oracle.py, the replay the GPU ISS keypoints (csrc/iss.cu) are held to."""
import importlib.util
import os

import numpy as np
import pytest

import iss_oracle as O

# synth.py is plain numpy; load it by path so these tests do not need the CUDA library behind the package
_spec = importlib.util.spec_from_file_location("ri_synth", os.path.join(
    os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
    "point-cloud-registration-based-on-rotation-invariant-feature_b200", "synth.py"))
synth = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(synth)


@pytest.mark.parametrize("seed", [1, 2])
def test_oracle_equals_literal_open3d_loop(seed):
    clouds = synth.make_clouds(4, 200, seed=seed)
    for b in range(4):
        X = clouds[b, :3].T.copy()
        for kw in ({}, dict(salient_radius=0.3, non_max_radius=0.2, min_neighbors=8)):
            o = O.iss(X, **kw)
            kp, third = O.iss_literal(X, **kw)
            amb = o['amb']
            assert amb.mean() < 0.2
            assert set(o['idx'][~amb[o['idx']]]) == set(kp[~amb[kp]])
            clear = ~amb
            assert np.allclose(o['saliency'][clear], third[clear], rtol=0, atol=1e-9 * np.abs(o['e1']).max())


def test_resolution_formula():
    rng = np.random.default_rng(0)
    X = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
    X[7] = X[3]                                                 # a duplicate contributes 0 twice
    d = np.full((300, 300), np.inf)
    for i in range(300):
        d[i] = O.fp32_dist(np.repeat(X[i:i + 1], 300, 0), X)
        d[i, i] = np.inf
    want = np.sqrt(d.min(1)).mean()
    res, n = O.resolution(X)
    assert n == 300 and abs(res - want) <= 1e-14 * want
    assert d[3].min() == 0 and d[7].min() == 0
    rs, rnm = O.auto_radii(X)
    assert rs == np.float32(6 * res) and rnm == np.float32(4 * res)
    Xn = X.copy(); Xn[5] = np.nan                               # non-finite points are not counted
    assert O.resolution(Xn)[1] == 299
    assert O.resolution(X[:1]) == (0.0, 0)


def test_duplicates_are_both_kept():
    X = synth.make_clouds(1, 400, seed=4)[0, :3].T.copy()
    o = O.iss(X)
    k = int(o['idx'][np.argmax(o['saliency'][o['idx']])])
    Y = np.concatenate([X, X[k:k + 1]], 0)
    oy = O.iss(Y, *o['radii'])
    assert k in oy['idx'] and 400 in oy['idx']
    assert oy['saliency'][k] == oy['saliency'][400]
    assert not oy['amb'][k]


def test_exact_plane_and_identical_points_give_none():
    rng = np.random.default_rng(1)
    P = np.zeros((500, 3), np.float32)
    P[:, :2] = rng.uniform(-1, 1, (500, 2))
    o = O.iss(P)
    assert len(o['idx']) == 0 and np.all(o['saliency'] == 0)
    o = O.iss(np.full((64, 3), 0.25, np.float32))
    assert len(o['idx']) == 0 and o['radii'] == (0, 0)
    o = O.iss(np.full((64, 3), 0.25, np.float32), 0.1, 0.1)     # explicit radii: C is zero
    assert len(o['idx']) == 0 and np.all(o['saliency'] == 0)


def test_min_neighbors_boundaries():
    X = synth.make_clouds(1, 300, seed=5)[0, :3].T.copy()
    o = O.iss(X, 0.3, 0.2, min_neighbors=1)
    cs, cn = o['count_s'], o['count_nm']
    m = int(np.median(cs))
    om = O.iss(X, 0.3, 0.2, min_neighbors=m)
    assert np.all(om['saliency'][cs < m] == 0)
    assert np.array_equal(om['saliency'][cs >= m], o['saliency'][cs >= m])
    assert np.all(cn[om['idx']] >= m)
    # a keypoint at min_neighbors = 1 whose suppression radius holds exactly c points stays one up to c and not beyond
    k = [int(i) for i in o['idx'] if cs[i] >= cn[i] + 1 and not o['amb'][i]]
    assert k
    c = int(cn[k[0]])
    assert k[0] in O.iss(X, 0.3, 0.2, min_neighbors=c)['idx']
    assert k[0] not in O.iss(X, 0.3, 0.2, min_neighbors=c + 1)['idx']


def test_box_keypoints_lie_on_edges_and_cover_the_corners():
    rng = np.random.default_rng(3)
    h = np.array([0.8, 0.6, 0.4]); n = 4000
    area = np.array([h[1] * h[2], h[0] * h[2], h[0] * h[1]])
    axis = rng.choice(3, size=n, p=area / area.sum())
    sign = rng.choice([-1.0, 1.0], size=n)
    p = rng.uniform(-1, 1, (n, 3)) * h
    p[np.arange(n), axis] = sign * h[axis]
    X = p.astype(np.float32)
    o = O.iss(X)
    rs = float(o['radii'][0])
    kp = X[o['idx']].astype(np.float64)
    assert len(kp) >= 8
    # face interiors are exact planes (e3 = 0): every keypoint is within r_s of an edge (two coordinates near +-h)
    edge_gap = np.sort(np.abs(np.abs(kp) - h), axis=1)[:, 1]
    assert edge_gap.max() <= rs
    # and every corner has a keypoint nearby
    corners = np.array([[sx * h[0], sy * h[1], sz * h[2]] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)])
    assert np.linalg.norm(kp[:, None] - corners[None], axis=2).min(0).max() <= 1.25 * rs
