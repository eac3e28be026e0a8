"""The colored-ICP reference (tests/icp_colored_reference.py) checked on its own, and the bindings' own argument checks: no
device needed."""
import numpy as np
import pytest

import icp_colored_reference as cref
import icp_plane_reference as pref
from cwipc_util_b200 import synthetic
from icp_colored_reference import RAMP_COLOURS, RAMP_SPACING, ramp, revolution_pair

DT = synthetic.cwipc_point_numpy_dtype


def rot_deg(T):
    R = np.asarray(T)[:3, :3]
    return float(np.degrees(np.arccos(np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0))))


def test_intensity_is_the_exact_colour_sum_over_765():
    pts = np.zeros(4, DT)
    pts["r"], pts["g"], pts["b"], pts["tile"] = [0, 255, 1, 100], [0, 255, 2, 0], [0, 255, 3, 7], [9, 9, 9, 9]
    assert list(cref.intensity(pts)) == [0.0, 1.0, 6.0 / 765.0, 107.0 / 765.0]


def test_a_linear_colour_ramp_gives_its_gradient_orthogonal_to_the_normal():
    for colour in RAMP_COLOURS:
        pts, want = ramp(colour=colour)
        P = cref.xyz32(pts)
        nrm = pref.estimate_normals(P, 3 * RAMP_SPACING, 30).normals
        assert np.all(nrm[:, :2] == 0.0) and np.all(np.abs(nrm[:, 2]) == 1.0)
        g = cref.color_gradients(P, cref.intensity(pts), nrm, 3 * RAMP_SPACING, 30)
        # the float64 solution is within a few float64 ulps of the true gradient, so it rounds to the same float32
        assert np.all(g == want.astype(np.float32)), (colour, np.abs(g - want).max())
        assert np.all(g[:, 2] == 0.0)


def test_fewer_than_4_neighbours_or_a_zero_normal_gives_zero():
    pts, _ = ramp(n=10)
    P = cref.xyz32(pts)
    inten = cref.intensity(pts)
    nrm = pref.estimate_normals(P, 1.5 * RAMP_SPACING, 30).normals
    g = cref.color_gradients(P, inten, nrm, 1.5 * RAMP_SPACING, 30)
    assert np.all(np.any(g != 0.0, axis=1))
    # a radius that only reaches the 4 face neighbours: the corners have 3 points (themselves and 2 neighbours)
    g = cref.color_gradients(P, inten, nrm, 1.0 * RAMP_SPACING, 30)
    count = (pref.neighbourhoods(P, 1.0 * RAMP_SPACING, 30) >= 0).sum(1)
    assert np.all(g[count < 4] == 0.0) and np.any(count < 4) and np.all(np.any(g[count >= 4] != 0.0, axis=1))
    g = cref.color_gradients(P, inten, np.zeros_like(nrm), 3 * RAMP_SPACING, 30)
    assert np.all(g == 0.0)


def test_lambda_one_is_the_point_to_plane_step():
    rng = np.random.default_rng(3)
    p, q = rng.normal(size=(500, 3)), rng.normal(size=(500, 3))
    nrm = rng.normal(size=(500, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    grad, Is, It = rng.normal(size=(500, 3)), rng.uniform(size=500), rng.uniform(size=500)
    o = np.array([0.1, 0.2, -0.3])
    assert np.array_equal(cref.colored_step(p, q, nrm, grad, Is, It, o, 1.0), pref.plane_step(p, q, nrm, o))
    assert not np.array_equal(cref.colored_step(p, q, nrm, grad, Is, It, o, 0.968), pref.plane_step(p, q, nrm, o))


@pytest.mark.parametrize("y_degrees", [3.0, 6.0])
def test_colored_icp_recovers_the_turn_point_to_plane_misses(y_degrees):
    source, target, P = revolution_pair(y_degrees)
    plane = pref.icp_point_to_plane(source, target, 0.05, 0.04)
    colored = cref.icp_colored(source, target, 0.05, 0.04)
    print(f"{y_degrees} deg: point-to-plane {plane.iterations} iterations, {rot_deg(plane.matrix @ P):.3f} deg; "
          f"colored {colored.iterations} iterations, {rot_deg(colored.matrix @ P):.4f} deg")
    assert rot_deg(plane.matrix @ P) > 3.0
    assert rot_deg(colored.matrix @ P) < 0.1
    assert colored.fitness > 0.99


class _NoCloud:
    """Stands in for a cloud; the binding must reject init before it asks for the cloud's pointer."""

    def as_cwipc_p(self):
        raise AssertionError("the library was called")


@pytest.mark.parametrize("init", [np.eye(3), np.eye(4)[:3], np.zeros(16), np.zeros((4, 4, 1)), [[1, 0, 0, 0]] * 5])
def test_binding_rejects_a_wrong_init_shape_before_the_library(init):
    from cwipc_util_b200 import util
    with pytest.raises(ValueError):
        util.cwipc_icp_colored(_NoCloud(), _NoCloud(), 0.05, 0.02, init=init)


def test_bindings_are_declared():
    from cwipc_util_b200 import util
    assert {"cwipc_icp_colored", "cwipc_estimate_color_gradients"} <= set(util.__all__)
    assert callable(util.cwipc_icp_colored) and callable(util.cwipc_estimate_color_gradients)
