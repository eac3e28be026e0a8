"""The point-to-plane reference (tests/icp_plane_reference.py) checked on its own, and the bindings' own argument checks: no
device needed."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import icp_plane_reference as pref


def pose(seed, degrees, metres):
    """A seeded rigid motion: a rotation of `degrees` about a random axis and a translation of `metres`."""
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3)
    T = np.eye(4)
    T[:3, :3] = Rotation.from_rotvec(np.radians(degrees) * axis / np.linalg.norm(axis)).as_matrix()
    t = rng.normal(size=3)
    T[:3, 3] = metres * t / np.linalg.norm(t)
    return T


def sheet(n, seed):
    """A wavy 2 m x 2 m sheet: no motion slides it along itself."""
    rng = np.random.default_rng(seed)
    u, v = rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)
    return np.stack([u, 0.3 * np.sin(3 * u) * np.cos(2 * v) + 0.1 * u * v, v], 1).astype(np.float32)


def lattice(n, spacing=1.0):
    return (np.stack(np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij"), -1).reshape(-1, 3) * spacing).astype(np.float32)


def test_normals_of_a_tilted_plane_and_of_a_sphere():
    rng = np.random.default_rng(1)
    R = Rotation.from_rotvec([0.3, -0.5, 0.2]).as_matrix()
    uv = rng.uniform(-1, 1, (20000, 2))
    plane = (np.c_[uv, np.zeros(len(uv))] @ R.T + [0.5, 2.0, -1.0]).astype(np.float32)
    got = pref.estimate_normals(plane, 0.05, 30)
    assert np.all(got.count >= 3)
    assert np.abs(np.abs(got.normals.astype(np.float64) @ R[:, 2]) - 1.0).max() < 1e-5
    d = rng.normal(size=(30000, 3))
    sphere = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    got = pref.estimate_normals(sphere, 0.05, 30)
    radial = sphere.astype(np.float64) / np.linalg.norm(sphere.astype(np.float64), axis=1, keepdims=True)
    assert np.abs(np.einsum("na,na->n", got.normals.astype(np.float64), radial)).min() > 1 - 1e-3


def test_zero_normals_for_isolated_points_pairs_and_coincident_points():
    isolated = np.float32([[0, 0, 0], [1, 0, 0], [0, 1, 0]])
    pair = np.float32([[5, 5, 5], [5.01, 5, 5]])
    same = np.repeat(np.float32([[-3, 2, 1]]), 6, axis=0)
    spread = np.float32([[10, 10, 10], [10.01, 10, 10], [10, 10.01, 10], [10, 10, 10.01]])
    got = pref.estimate_normals(np.concatenate([isolated, pair, same, spread]), 0.1, 30)
    assert np.array_equal(got.count, [1, 1, 1, 2, 2, 6, 6, 6, 6, 6, 6, 4, 4, 4, 4])
    assert np.all(got.normals[:11] == 0.0)
    assert np.all(np.linalg.norm(got.normals[11:], axis=1) > 0.99)


def test_neighbourhood_ties_go_to_the_lower_index():
    g = lattice(7)
    order = np.random.default_rng(3).permutation(len(g))
    pts = g[order]
    # the 6 face neighbours of an inner point are all at d2 = 1: with max_nn = 4 only the 3 of smallest index join it
    nb = pref.neighbourhoods(pts, 1.0, 4)
    d2 = pref.d2f(pts[:, None, :], pts[np.maximum(nb, 0)])
    inner = np.flatnonzero(np.all((pts >= 1) & (pts <= 5), axis=1))
    for i in inner:
        faces = np.flatnonzero(pref.d2f(pts[i][None, :], pts) == 1.0)
        assert len(faces) == 6
        assert nb[i, 0] == i and d2[i, 0] == 0.0
        assert list(nb[i, 1:]) == sorted(faces)[:3]


def test_neighbourhoods_are_the_brute_force_ones():
    rng = np.random.default_rng(4)
    pts = (rng.integers(0, 12, (3000, 3)) * 0.25).astype(np.float32)   # many exact duplicates and ties
    for max_nn in (3, 8, 32):
        nb = pref.neighbourhoods(pts, 0.6, max_nn)
        d2 = pref.d2f(pts[:, None, :], pts[None, :, :])
        for i in range(0, len(pts), 97):
            ok = np.flatnonzero(d2[i] <= pref.limit32(0.6))
            want = ok[np.lexsort((ok, d2[i][ok]))][:max_nn]
            assert list(nb[i][nb[i] >= 0]) == list(want)


def test_one_step_with_exact_pairs_is_first_order_and_the_loop_recovers_the_motion():
    target = sheet(20000, 1)
    nrm = pref.estimate_normals(target, 0.08, 30).normals
    assert np.all(np.linalg.norm(nrm, axis=1) > 0.99)
    T0 = pose(2, 0.5, 0.005)
    source = pref.move(target, np.linalg.inv(T0))   # target = T0 * source, up to the float32 rounding of the source
    dT = pref.plane_step(source, target, nrm, pref.box_centre(target))
    err = dT @ np.linalg.inv(T0)
    assert np.degrees(np.arccos(np.clip((np.trace(err[:3, :3]) - 1) / 2, -1, 1))) < np.degrees(1e-4)
    assert np.abs(err[:3, 3]).max() < 1e-4
    r = pref.icp_point_to_plane(source, target, 0.05, 0.08, max_iterations=60, relative_fitness=0.0, relative_rmse=0.0)
    assert r.correspondences == len(source)
    assert np.abs(r.matrix - T0).max() < 1e-9, np.abs(r.matrix - T0).max()


def test_on_a_flat_plane_the_unseen_components_are_exactly_zero():
    rng = np.random.default_rng(5)
    q = np.c_[rng.uniform(-1, 1, (5000, 2)), np.zeros(5000)].astype(np.float32)
    p = (q + np.float32([0.01, -0.02, 0.003])).astype(np.float32)      # slid along the plane and lifted off it
    nrm = np.tile(np.float32([0, 0, 1]), (len(q), 1))
    o = pref.box_centre(q)
    A_J = np.concatenate([np.cross(p - o, nrm), nrm], 1)
    x = pref.min_norm_solve(A_J.T @ A_J, -(A_J.T @ np.einsum("na,na->n", (p - q).astype(np.float64), nrm)))
    assert x[2] == 0.0 and x[3] == 0.0 and x[4] == 0.0                    # turn about the normal, slide along the plane
    assert abs(x[5] + 0.003) < 1e-9
    dT = pref.plane_step(p, q, nrm, o)
    assert np.all(np.isfinite(dT))
    # (alpha and beta are rounding-sized, not exactly 0, so Ry Rx adds their product to the in-plane terms)
    assert max(abs(dT[0, 1]), abs(dT[1, 0]), abs(dT[0, 3]), abs(dT[1, 3])) < 1e-15
    assert abs(dT[2, 3] + 0.003) < 1e-9
    # a system with no normal at all gives the identity
    assert np.array_equal(pref.plane_step(p, q, np.zeros_like(nrm), o), np.eye(4))


def test_euler_matrix_is_rz_ry_rx():
    x = np.array([0.1, -0.2, 0.3, 1.0, 2.0, 3.0])
    R = Rotation.from_euler("ZYX", [0.3, -0.2, 0.1]).as_matrix()
    T = pref.euler_matrix(x)
    assert np.abs(T[:3, :3] - R).max() < 1e-15 and np.array_equal(T[:3, 3], x[3:])


class _NoCloud:
    """Stands in for a cloud; the binding must reject init before it asks for the cloud's pointer."""

    def as_cwipc_p(self):
        raise AssertionError("the library was called")


@pytest.mark.parametrize("init", [np.eye(3), np.eye(4)[:3], np.zeros(16), np.zeros((4, 4, 1)), [[1, 0, 0, 0]] * 5])
def test_binding_rejects_a_wrong_init_shape_before_the_library(init):
    from cwipc_util_b200 import util
    with pytest.raises(ValueError):
        util.cwipc_icp_point_to_plane(_NoCloud(), _NoCloud(), 0.05, 0.02, init=init)


def test_bindings_are_declared():
    from cwipc_util_b200 import util
    assert {"cwipc_icp_point_to_plane", "cwipc_estimate_normals"} <= set(util.__all__)
