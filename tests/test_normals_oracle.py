"""CPU self-test of the normal-estimation reference (tests/normals_oracle.py, row f6): exact on a plane, radial on a sphere
within the curvature bound, the (0,0,1) default, and both orientation rules.  No GPU needed."""
import numpy as np

import normals_oracle as ref


def _angle(a, b):
    """Angle in radians between the rows of a and b, ignoring the sign."""
    c = np.abs(np.sum(a * b, 1)) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))
    return np.arccos(np.clip(c, 0.0, 1.0))


def test_plane_normal_is_exact():
    rng = np.random.default_rng(1)
    n = np.array([1.0, 2.0, 2.0]) / 3.0
    u = np.cross(n, [1.0, 0, 0]); u /= np.linalg.norm(u); v = np.cross(n, u)
    uv = rng.uniform(-1, 1, (2000, 2))
    xyz = 0.3 * n + uv[:, :1] * u + uv[:, 1:] * v
    nrm, count = ref.estimate_normals(xyz, 0.2, 30)
    assert (count >= 3).all() and np.median(count) == 30
    assert _angle(nrm, np.tile(n, (len(xyz), 1))).max() < 1e-7


def test_sphere_normal_is_radial_within_curvature_bound():
    rng = np.random.default_rng(2)
    R, r = 1.0, 0.2
    p = rng.standard_normal((4000, 3)); p /= np.linalg.norm(p, axis=1, keepdims=True)
    xyz = R * p
    nrm, count = ref.estimate_normals(xyz, r, 30)
    assert (count >= 3).all()
    # every neighbour lies within r of q, i.e. within the angle asin(r/R) of it on the sphere: the fitted plane cannot
    # tilt further than that from the tangent plane at q
    assert _angle(nrm, p).max() <= np.arcsin(r / R)
    assert np.median(_angle(nrm, p)) < 0.02


def test_fewer_than_three_neighbours_give_default():
    rng = np.random.default_rng(3)
    xyz = rng.uniform(0, 10, (200, 3))                       # spacing ~1.7: a radius of 0.01 leaves each point alone
    nrm, count = ref.estimate_normals(xyz, 0.01, 30)
    assert (count == 1).all() and (nrm == [0.0, 0.0, 1.0]).all()
    idx = np.tile(np.arange(3), (3, 1))
    nrm, _, _ = ref.normals_from_neighbours(xyz[:3], idx, np.array([2, 2, 2]))
    assert (nrm == [0.0, 0.0, 1.0]).all()
    same = np.zeros((5, 3))                                  # coincident points: zero trace
    nrm, _ = ref.estimate_normals(same, 1.0, 5)
    assert (nrm == [0.0, 0.0, 1.0]).all()
    nrm, _ = ref.estimate_normals(same, 1.0, 5, camera=np.array([0.0, 0.0, -1.0]))
    assert (nrm == [0.0, 0.0, -1.0]).all()                   # the default is oriented too


def test_orientation_rules():
    rng = np.random.default_rng(4)
    uv = rng.uniform(-1, 1, (1000, 2))
    xyz = np.c_[uv, np.zeros(1000)]                          # the plane z = 0
    up, _ = ref.estimate_normals(xyz, 0.2, 20, camera=np.array([0.0, 0.0, 5.0]))
    down, _ = ref.estimate_normals(xyz, 0.2, 20, camera=np.array([0.0, 0.0, -5.0]))
    assert np.allclose(up, [0, 0, 1]) and np.allclose(down, [0, 0, -1])
    prior = np.tile([0.1, -0.2, -1.0], (1000, 1))
    p, _ = ref.estimate_normals(xyz, 0.2, 20, prior=prior)
    assert np.allclose(p, [0, 0, -1])
    prior[::2] *= -1
    p, _ = ref.estimate_normals(xyz, 0.2, 20, prior=prior)
    assert np.allclose(p[::2], [0, 0, 1]) and np.allclose(p[1::2], [0, 0, -1])
