"""The ICP reference (tests/icp_reference.py) checked on its own, and the binding's own argument check: no device needed."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import icp_reference as ref


def pose(seed, degrees, metres):
    """A seeded rigid motion: a rotation of `degrees` about a random axis and a translation of `metres`."""
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3)
    T = np.eye(4)
    T[:3, :3] = Rotation.from_rotvec(np.radians(degrees) * axis / np.linalg.norm(axis)).as_matrix()
    t = rng.normal(size=3)
    T[:3, 3] = metres * t / np.linalg.norm(t)
    return T


def surface(n, seed):
    """Points on a wavy sheet with some depth structure, 2 m x 2 m: a shape ICP can lock onto."""
    rng = np.random.default_rng(seed)
    u, v = rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)
    return np.stack([u, v, 0.3 * np.sin(3 * u) * np.cos(2 * v) + 0.1 * u * v], 1).astype(np.float32)


def test_recovers_a_seeded_motion_of_a_noiseless_cloud():
    target = surface(20000, 1)
    T0 = pose(2, 2.0, 0.01)
    source = ref.move(target, np.linalg.inv(T0))   # target = T0 * source, up to the float32 rounding of the source
    r = ref.icp(source, target, 0.05, max_iterations=60, relative_fitness=0.0, relative_rmse=0.0)
    assert r.correspondences == len(source)
    assert np.abs(r.matrix - T0).max() < 1e-9, np.abs(r.matrix - T0).max()
    assert r.inlier_rmse < 1e-7


def test_one_step_solve_agrees_with_scipy_align_vectors():
    rng = np.random.default_rng(3)
    p = rng.normal(size=(5000, 3)) * [1.0, 0.5, 0.2] + [3.0, -2.0, 1.0]
    T0 = pose(4, 7.0, 0.2)
    q = p @ T0[:3, :3].T + T0[:3, 3] + rng.normal(size=p.shape) * 0.01
    T = ref.kabsch(p, q)
    pc, qc = p - p.mean(0), q - q.mean(0)
    R, _ = Rotation.align_vectors(qc, pc)            # R minimises sum |qc_i - R pc_i|^2
    assert np.abs(T[:3, :3] - R.as_matrix()).max() < 1e-12
    assert np.abs(T[:3, 3] - (q.mean(0) - R.as_matrix() @ p.mean(0))).max() < 1e-12
    assert abs(np.linalg.det(T[:3, :3]) - 1.0) < 1e-12


def test_a_reflection_is_never_returned():
    rng = np.random.default_rng(5)
    p = rng.normal(size=(200, 3))
    q = p * [1.0, 1.0, -1.0]                         # the best orthogonal map is a mirror; Kabsch must keep det +1
    T = ref.kabsch(p, q)
    assert abs(np.linalg.det(T[:3, :3]) - 1.0) < 1e-12


def test_ties_go_to_the_lower_index():
    # a lattice with spacing 1, listed in a shuffled order; every query sits exactly half way between two lattice points
    # along x, so the two float32 d2 are equal and only the index decides
    g = np.stack(np.meshgrid(np.arange(6), np.arange(6), np.arange(6), indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    order = np.random.default_rng(6).permutation(len(g))
    target = g[order]
    queries = (g[g[:, 0] < 5] + np.float32([0.5, 0.0, 0.0])).astype(np.float32)
    idx, d2 = ref.Matcher(target).nearest(queries, np.float32(1.0))
    pos = np.empty(len(g), np.int64)
    pos[order] = np.arange(len(g))                   # pos[lattice point] = its index in the target
    key = lambda p: (p[:, 0].astype(np.int64) * 6 + p[:, 1].astype(np.int64)) * 6 + p[:, 2].astype(np.int64)
    left, right = pos[key(queries - [0.5, 0, 0])], pos[key(queries + [0.5, 0, 0])]
    assert np.all(d2 == np.float32(0.25))
    assert np.array_equal(idx, np.minimum(left, right))
    assert np.any(left < right) and np.any(right < left)


def test_bound_is_inclusive_and_taken_in_float32():
    target = np.float32([[0.0, 0.0, 0.0]])
    lim = ref.limit32(0.5)
    q = np.float32([[0.5, 0.0, 0.0], [np.nextafter(np.float32(0.5), np.float32(1)), 0.0, 0.0]])
    idx, d2 = ref.Matcher(target).nearest(q, lim)
    assert list(idx) == [0, -1]


def test_empty_clouds_and_no_correspondences():
    pts = surface(100, 7)
    init = pose(8, 1.0, 0.01)
    for s, t in ((pts[:0], pts), (pts, pts[:0])):
        r = ref.icp(s, t, 0.1, init=init)
        assert r.correspondences == 0 and r.iterations == 0 and r.fitness == 0.0 and r.inlier_rmse == 0.0
        assert np.array_equal(r.matrix, init)
    r = ref.icp(pts + np.float32(10.0), pts, 0.1)
    assert r.correspondences == 0 and r.iterations == 0 and np.array_equal(r.matrix, np.eye(4))


class _NoCloud:
    """Stands in for a cloud; the binding must reject init before it asks for the cloud's pointer."""

    def as_cwipc_p(self):
        raise AssertionError("the library was called")


@pytest.mark.parametrize("init", [np.eye(3), np.eye(4)[:3], np.zeros(16), np.zeros((4, 4, 1)), [[1, 0, 0, 0]] * 5])
def test_binding_rejects_a_wrong_init_shape_before_the_library(init):
    from cwipc_util_b200 import util
    with pytest.raises(ValueError):
        util.cwipc_icp(_NoCloud(), _NoCloud(), 0.05, init=init)
